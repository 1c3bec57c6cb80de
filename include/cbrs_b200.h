/* cbrs_b200.h - C ABI of the B200 (sm_100a) hot path of Deep_CBRS_Amar_Renaissance.
 *
 * Path: graph build -> GNN propagation (GCN / LightGCN / GraphSAGE / GAT / relational)
 *       -> gather user+item rows (+ content rows) -> dense MLP -> sigmoid -> top-k.
 *
 * The reference (pure Python on TensorFlow + Spektral) has no FFI: its "operator
 * API" is the Python layer / model call convention (SURVEY.md section 8b).  Each entry
 * point below names the reference lines whose work it replaces; INTEGRATION.md
 * shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in _host;
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it,
 *    never synchronise, never allocate: scratch comes from the caller, sized by
 *    the matching *_workspace_bytes query (host-only, no CUDA call);
 *  - returns 0 on success, <0 on error (CBRS_E_*); the message is kept per host
 *    thread and read with cbrs_last_error();
 *  - feature matrices are row-major float32 with an explicit leading dimension
 *    (ld, in elements) so layers write straight into column slices of one
 *    [N, D_out] buffer (the 'concatenation' reduction costs nothing);
 *  - row pointers are int64, column ids int32 (2e9 + 1.1e7 edges still fit).
 */
#ifndef CBRS_B200_H_
#define CBRS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CBRS_OK 0
#define CBRS_E_INVALID (-1)   /* bad argument */
#define CBRS_E_WORKSPACE (-2) /* workspace too small */
#define CBRS_E_CUDA (-3)      /* CUDA runtime error (launch failed, wrong device, ...) */
#define CBRS_E_UNSUPPORTED (-4)

/* ---- library ---------------------------------------------------------- */
int cbrs_version(void);
const char *cbrs_last_error(void);
/* 0 when the current CUDA device is compute capability 10.x (the only target). */
int cbrs_check_device(void);

/* ---- graph build (rows G1-G3) ------------------------------------------
 * Replaces, on device: scipy COO->CSR + duplicate summing + spektral gcn_filter
 * (call sites /root/reference/src/models/gnn.py:283, src/layers/lightgcn_conv.py:58)
 * and the tf.sparse.reorder of src/utilities/math.py:47-56.
 * Stable LSD radix sort of (row,col) keys, run-length duplicate sum, row-pointer
 * scan, symmetric normalisation.  Bit-exact structure vs. the oracle.          */
#define CBRS_GRAPH_DEDUP_SUM 1      /* sum duplicate (row,col) entries in input order        */
#define CBRS_GRAPH_ADD_SELF_LOOPS 2 /* M_ii += 1 (entry created if absent); needs DEDUP_SUM  */
#define CBRS_GRAPH_SYM_NORM 4       /* vals = fl32(fl32(d_i*m_ij)*d_j), d = rowsum^-1/2      */
#define CBRS_GRAPH_DROP_DIAG 8      /* drop (i,i) entries before anything else (GAT edge set) */

size_t cbrs_graph_build_workspace_bytes(int64_t nnz, int64_t n_nodes, int flags);
/* Capacity of colidx / vals must be nnz (+ n_nodes with ADD_SELF_LOOPS).
 * rowptr has n_nodes+1 entries; the output edge count is rowptr[n_nodes]
 * (also written to *nnz_out, a device int64, if not NULL).
 * coo_val may be NULL (all ones).                                              */
int cbrs_graph_build_csr(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val,
                         int64_t nnz, int64_t n_nodes, int flags, int64_t *rowptr,
                         int32_t *colidx, float *vals, int64_t *nnz_out, void *workspace,
                         size_t workspace_bytes, void *stream);

/* Relational variant (row R, extension): rel[e] in [0,n_rel) joins the key as
 * (row, rel, col); the output column id is rel*n_nodes + col so one SpMM over the
 * stacked per-relation transforms [n_rel*N, H] does the grouped scatter.
 * Self loops (ADD_SELF_LOOPS) are tagged with relation self_rel.  Normalisation uses the
 * node degree over ALL relations, so the values equal gcn_filter(A)'s and n_rel = 1
 * reproduces cbrs_graph_build_csr exactly.                                        */
int cbrs_graph_build_csr_rel(const int32_t *coo_row, const int32_t *coo_col, const int32_t *coo_rel,
                             const float *coo_val, int64_t nnz, int64_t n_nodes, int32_t n_rel,
                             int32_t self_rel, int flags, int64_t *rowptr, int32_t *colidx, float *vals,
                             int64_t *nnz_out, void *workspace, size_t workspace_bytes, void *stream);

/* ---- partitioned build: the rows [row_lo, row_hi) of the graph cbrs_graph_build_csr builds -------------------
 * A rank of a row partition builds only its own row blocks, bit for bit the rows the whole build gives them:
 *   1. cbrs_coo_row_histogram over every piece of the COO -> exact entry counts per row (cuts, buffer sizes);
 *   2. cbrs_coo_select_rows over every piece, in input order -> the block's entries, in their input order (the
 *      duplicate sum adds them in that order);
 *   3. cbrs_graph_build_block: sort, duplicate sum, self loops and row pointer for the block's rows only.  With
 *      CBRS_GRAPH_SYM_NORM it writes the block's d_i = fl32(1/sqrt(double(rowsum_i))) to dinv_out and leaves the
 *      values UNscaled: d_j of most columns belongs to other blocks;
 *   4. cbrs_graph_block_scale once every block's d is known: vals = fl32(fl32(d_i*m_ij)*d_j), d = the full vector.
 * Same kernels and rounding as cbrs_graph_build_csr, so rowptr / colidx / vals equal that build's rows row_lo..row_hi
 * (rowptr rebased to 0, global column ids).  The workspace scales with the block's entries.                     */
/* counts[r] += entries of row r, r in [0, n_rows) (int64, caller zeroes it; other rows are ignored) */
int cbrs_coo_row_histogram(const int32_t *coo_row, int64_t n, int64_t n_rows, int64_t *counts, void *stream);
size_t cbrs_coo_select_rows_workspace_bytes(int64_t n);
/* Appends the entries with row_lo <= row < row_hi, in input order, at out[*cursor ..] and advances *cursor (device
 * int64) by their number; rebase != 0 stores row - row_lo.  coo_val / out_val may be NULL.  Entries that would land
 * at or past `capacity` are not written (the cursor still counts them: compare it with the capacity afterwards).  */
int cbrs_coo_select_rows(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val, int64_t n,
                         int64_t row_lo, int64_t row_hi, int rebase, int32_t *out_row, int32_t *out_col,
                         float *out_val, int64_t *cursor, int64_t capacity, void *workspace, size_t workspace_bytes,
                         void *stream);
/* nnz = the block's entries (global row ids); n_rows = row_hi - row_lo; n_cols = the graph's node count.
 * Capacity of colidx / vals: nnz (+ n_rows with ADD_SELF_LOOPS).  rowptr [n_rows + 1].  dinv_out [n_rows] (needed
 * with SYM_NORM).                                                                                              */
size_t cbrs_graph_build_block_workspace_bytes(int64_t nnz, int64_t n_rows, int flags);
int cbrs_graph_build_block(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val, int64_t nnz,
                           int64_t row_lo, int64_t row_hi, int64_t n_cols, int flags, int64_t *rowptr,
                           int32_t *colidx, float *vals, float *dinv_out, int64_t *nnz_out, void *workspace,
                           size_t workspace_bytes, void *stream);
/* rows [row_lo, row_lo + n_rows) of a block built above; dinv: all n_cols degrees */
int cbrs_graph_block_scale(const int64_t *rowptr, const int32_t *colidx, float *vals, int64_t n_rows, int64_t row_lo,
                           int64_t n_cols, const float *dinv, void *stream);

/* ---- work decomposition -------------------------------------------------
 * Rows are cut into chunks of at most chunk_edges edges so that power-law item
 * rows do not serialise on one warp.  A row with a single chunk is written by
 * the chunk kernel itself; a row with several ("heavy") parks one partial per
 * chunk and is summed in ascending chunk order by a second kernel: a fixed
 * reduction tree, so results do not depend on launch shape or on how rows are
 * partitioned over GPUs.                                                        */
typedef struct cbrs_csr {
    int64_t n_rows;            /* rows held here (a rank's slice in the multi-GPU case)   */
    int64_t nnz;
    const int64_t *rowptr;     /* [n_rows+1], offsets into colidx/vals                    */
    const int32_t *colidx;     /* [nnz] global column ids, ascending inside a row         */
    const float *vals;         /* [nnz] or NULL (all ones)                                */
    int32_t chunk_edges;       /* max edges per chunk                                     */
    int64_t n_chunks;
    const int32_t *chunk_row;  /* [n_chunks] local row of the chunk                       */
    const int64_t *chunk_begin;/* [n_chunks] first edge; end = min(begin+chunk_edges,row end) */
    const int32_t *chunk_slot; /* [n_chunks] partial slot, or -1 when the row has one chunk */
    int64_t n_heavy;           /* rows with more than one chunk                           */
    const int32_t *heavy_row;  /* [n_heavy]                                               */
    const int64_t *heavy_slot_ptr; /* [n_heavy+1] slot range of each heavy row            */
    int64_t n_slots;
    const int32_t *chunk_len;  /* [n_chunks] edges of the chunk, or NULL: the rule given at chunk_begin. Set by the
                                  column-blocked decomposition below, whose chunks end at column-block borders     */
} cbrs_csr_t;

/* Pass 1: counts.  counts_out (device int64[3]) = {n_chunks, n_heavy, n_slots}. */
size_t cbrs_chunks_workspace_bytes(int64_t n_rows);
int cbrs_chunks_count(const int64_t *rowptr, int64_t n_rows, int32_t chunk_edges,
                      int64_t *counts_out, void *workspace, size_t workspace_bytes, void *stream);
/* Pass 2: fill (same workspace, untouched since pass 1). */
int cbrs_chunks_fill(const int64_t *rowptr, int64_t n_rows, int32_t chunk_edges, int32_t *chunk_row,
                     int64_t *chunk_begin, int32_t *chunk_slot, int32_t *heavy_row,
                     int64_t *heavy_slot_ptr, void *workspace, size_t workspace_bytes, void *stream);

/* Column-blocked decomposition (round 2: cuts the HBM traffic of the gather when the operand table [n_cols, D] is
 * larger than L2).  Rows with at least block_min_len edges are cut where their ascending column ids cross a multiple
 * of block_cols and then into pieces of at most chunk_edges edges; they are always "heavy" (partials merged in
 * ascending column order).  Their chunks follow all other rows' chunks in the list, ordered by (column block, row):
 * CTAs are dispatched in list order, so the resident warps gather from one window of block_cols operand rows that
 * stays in L2.  The cut points depend on the row's own column ids, block_cols and chunk_edges only => the reduction
 * tree of a row is the same on every launch shape and row partition.  chunk_len must be passed in cbrs_csr_t.
 * Replaces nothing in the reference (tf.sparse.sparse_dense_matmul, src/layers/lightgcn_conv.py:51-54, has no
 * schedule); counts_out as cbrs_chunks_count.  The count call synchronises the stream.                          */
size_t cbrs_chunks_blocked_workspace_bytes(int64_t n_rows, int64_t nnz, int64_t n_cols, int32_t block_min_len,
                                           int64_t block_cols);
int cbrs_chunks_blocked_count(const int64_t *rowptr, const int32_t *colidx, int64_t n_rows, int64_t nnz,
                              int64_t n_cols, int32_t chunk_edges, int32_t block_min_len, int64_t block_cols,
                              int64_t *counts_out, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_chunks_blocked_fill(const int64_t *rowptr, const int32_t *colidx, int64_t n_rows, int64_t nnz,
                             int64_t n_cols, int32_t chunk_edges, int32_t block_min_len, int64_t block_cols,
                             int32_t *chunk_row, int64_t *chunk_begin, int32_t *chunk_len, int32_t *chunk_slot,
                             int32_t *heavy_row, int64_t *heavy_slot_ptr, void *workspace,
                             size_t workspace_bytes, void *stream);

/* Row subset of a decomposition: the chunks of the rows listed in ids[0, n_ids) (duplicates allowed; ids outside
 * [0, n_rows) select nothing), in their original list order, with the needed heavy rows and their slots renumbered
 * compactly in the same order.  The result shares rowptr/colidx/vals/chunk_edges with g; a propagation kernel run on
 * it writes exactly the needed rows of Y, with the bits the full launch gives them.
 * Pass 1: counts_out (device int64[5]) = {n_chunks, n_heavy, n_slots, needed rows, their edges}.
 * Pass 2: fill (same workspace, untouched since pass 1); chunk_len is written when g has one, heavy_slot_ptr
 * [n_heavy + 1] must come zeroed.  The subset's spmm workspace is at most cbrs_spmm_workspace_bytes(g, d).        */
size_t cbrs_csr_subset_workspace_bytes(const cbrs_csr_t *g);
int cbrs_csr_subset_count(const cbrs_csr_t *g, const int64_t *ids, int64_t n_ids, int64_t *counts_out,
                          void *workspace, size_t workspace_bytes, void *stream);
int cbrs_csr_subset_fill(const cbrs_csr_t *g, int32_t *chunk_row, int64_t *chunk_begin, int32_t *chunk_len,
                         int32_t *chunk_slot, int32_t *heavy_row, int64_t *heavy_slot_ptr, void *workspace,
                         size_t workspace_bytes, void *stream);

/* ---- propagation kernels (rows P1, P2 aggregate, P4) ---------------------
 * Y[i, 0:D] = epilogue( reduce_j A_ij * X[col_j, 0:D] ), j over row i ascending.
 * Replaces tf.sparse.sparse_dense_matmul as invoked by spektral GCNConv /
 * ops.modal_dot (src/layers/lightgcn_conv.py:53) and the gather +
 * unsorted_segment_mean of GraphSageConv.                                       */
#define CBRS_AGG_WEIGHTED 0 /* sum of vals*x (vals NULL => sum of x)  */
#define CBRS_AGG_SUM 1      /* edge values ignored                      */
#define CBRS_AGG_MEAN 2     /* sum / edge count; empty row -> 0         */
#define CBRS_DTYPE_F32 0
#define CBRS_DTYPE_BF16 1   /* X stored bf16 (ldx in elements), products and accumulation fp32, Y fp32: the gathered
                               operand costs 2 B per element instead of 4 (264 instead of 520 B per edge at D=128) */

size_t cbrs_spmm_workspace_bytes(const cbrs_csr_t *g, int32_t d);
int cbrs_spmm_csr(const cbrs_csr_t *g, const void *x, int64_t ldx, void *y, int64_t ldy, int32_t d,
                  int agg, const float *bias, int relu, int dtype, void *workspace,
                  size_t workspace_bytes, void *stream);

/* ---- fused GAT layer (row P3) ---------------------------------------------
 * z [N,H] = X W (from cbrs_dense with CBRS_ROWOP_ATTN), p = z.a_self (rows of this
 * slice), q = z.a_neigh (all nodes).  One pass per row: leaky-relu(0.2) edge
 * score, segment max, exp, sum (+1e-9), weighted aggregate, bias, relu.  The
 * edge set is the raw adjacency minus existing self loops plus (i,i), computed on
 * the fly; `row_offset` is the global id of local row 0.  Replaces spektral
 * GATConv._call_single (4 gathers + 3 segment ops).                              */
size_t cbrs_gat_workspace_bytes(const cbrs_csr_t *g, int32_t h);
int cbrs_gat_csr(const cbrs_csr_t *g, int64_t row_offset, const float *z, int64_t ldz,
                 const float *p, const float *q, float *y, int64_t ldy, int32_t h,
                 const float *bias, int relu, void *workspace, size_t workspace_bytes, void *stream);

/* ---- dense layer with fused gather + concat (rows P1 transform, P2, S1-S4) --
 * out[m, 0:n] = act( [ X1[idx1[m], 0:f1] || X2[idx2[m], 0:f2] ] @ W[f1+f2, n] + b )
 * idx* NULL => identity; X2 NULL => single source.  Keras Dense semantics
 * (kernel stored [in,out]); replaces tf.nn.embedding_lookup + Concatenate + Dense
 * of src/models/basic.py:31-37,72-75 and src/models/hybrid.py:72-89,136-140.    */
#define CBRS_ACT_NONE 0
#define CBRS_ACT_RELU 1
#define CBRS_ACT_SIGMOID 2
#define CBRS_ACT_TANH 3
#define CBRS_ROWOP_NONE 0
#define CBRS_ROWOP_L2NORM 1 /* v / sqrt(max(sum v^2, 1e-12)) before act (GraphSageConv)      */
#define CBRS_ROWOP_ATTN 2   /* also emit p = out.a_self, q = out.a_neigh (GATConv), n <= 128 */
int cbrs_dense(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2,
               int64_t ld2, const int64_t *idx2, int32_t f2, const float *w, const float *b,
               int64_t m, int32_t n, int act, int rowop, const float *a_self,
               const float *a_neigh, float *p_out, float *q_out, float *out, int64_t ldo,
               void *stream);

/* The same layer on the tensor cores (tcgen05, bf16 operands, fp32 accumulate): the tower GEMMs of the scorers
 * (src/models/hybrid.py:74-77: Dense 768 -> 256 -> 64 over the BERT rows; src/models/basic.py:33-34).
 * out = act( bf16([X1[idx1] || X2[idx2]]) @ bf16(W) + b ), out fp32.  W is handed over as the operand image that
 * cbrs_dense_tc_prepare writes from the Keras kernel [k, n] (cbrs_dense_tc_image_bytes(k, n) bytes, 16-byte
 * aligned; rewrite it whenever W changes).  Requirements: n <= 256, f1 and f2 multiples of 8, source rows 16-byte
 * aligned (ld % 4 == 0).  Results differ from cbrs_dense by the bf16 rounding of the operands only.          */
size_t cbrs_dense_tc_image_bytes(int32_t k, int32_t n);
int cbrs_dense_tc_prepare(const float *w, int32_t k, int32_t n, void *image, void *stream);
int cbrs_dense_tc(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2, int64_t ld2,
                  const int64_t *idx2, int32_t f2, const void *w_image, const float *b, int64_t m, int32_t n,
                  int act, float *out, int64_t ldo, void *stream);

/* The same layer over bf16-STORED sources, fed by TMA (the static content table of the hybrid models:
 * src/models/hybrid.py:136-140 gathers its rows by the batch's ids, hybrid.py:74-77 runs the towers on them).
 * cbrs_convert_f32_bf16 rounds a row-major fp32 matrix to bf16 once (round to nearest even: the rounding cbrs_dense_tc
 * applies to every row on every call, so both kernels multiply identical operands); k, ldx, ldo multiples of 4.
 * cbrs_dense_tc_bf16: X1 [rows1, ld1] and X2 [rows2, ld2] hold bf16 (ld in elements, % 8 == 0, 16-byte aligned bases);
 * rows of an indexed source arrive by cp.async.bulk.tensor tile::gather4, consecutive rows as one tiled box, W as
 * the image of cbrs_dense_tc_prepare; out_dtype = CBRS_DTYPE_F32 (float *out) or CBRS_DTYPE_BF16 (ldo in elements),
 * so a tower's layers chain without an fp32 round trip.  Requirements: f1, f2 multiples of 64, n <= 256, every index
 * in [0, rows), m <= rows when a source has no index.                                                               */
int cbrs_convert_f32_bf16(const float *x, int64_t ldx, int64_t m, int32_t k, void *out, int64_t ldo, void *stream);
int cbrs_dense_tc_bf16_eligible(int32_t f1, int32_t f2, int32_t n);
int cbrs_dense_tc_bf16(const void *x1, int64_t ld1, int64_t rows1, const int64_t *idx1, int32_t f1, const void *x2,
                       int64_t ld2, int64_t rows2, const int64_t *idx2, int32_t f2, const void *w_image,
                       const float *b, int64_t m, int32_t n, int act, void *out, int64_t ldo, int out_dtype,
                       void *stream);

/* Full-catalog scoring of the FEATURE-BASED hybrid scorer with a fused per-user top-k, chained on the tensor cores
 * (src/models/hybrid.py:72-89 for every (user, item) pair; the form all of econfigs/hybrid-gnn*.yaml use).  The caller
 * hoists what depends on one entity: the four towers and the first layer of dense3a / dense3b, split into a user half
 * (bias folded in) and an item half: P1 [U, c], Q1 [I, c] (collaborative branch), P2, Q2 (content branch), rows
 * contiguous.  Per pair the kernel computes, bf16 operands / fp32 accumulation, activations never leaving the SM:
 *   x1 = relu(relu(P1[u]+Q1[i]) w3a2 + b3a2),  x2 = relu(relu(P2[u]+Q2[i]) w3b2 + b3b2),
 *   g = relu([x1 || x2] wc1 + bc1),  score = sigmoid(relu(g wc2 + bc2) . wc3 + bc3)
 * w3a2, w3b2, wc2: [c, c]; wc1: [2c, c] (Keras [in, out], contiguous); c = 64.  ids_out [U, k] int32 item indices,
 * scores_out [U, k], descending, ties to the lower index; k <= 128.                                               */
size_t cbrs_score_hybrid_topk_bf16_workspace_bytes(void);
int cbrs_score_hybrid_topk_bf16(const float *P1, const float *Q1, const float *P2, const float *Q2, int64_t n_users,
                                int32_t n_items, int32_t c, const float *w3a2, const float *b3a2, const float *w3b2,
                                const float *b3b2, const float *wc1, const float *bc1, const float *wc2,
                                const float *bc2, const float *wc3, const float *bc3, int32_t k, int32_t *ids_out,
                                float *scores_out, void *workspace, size_t workspace_bytes, void *stream);
/* With per-user exclusion lists (contract above cbrs_score_catalog_topk_ex).  Null lists: cbrs_score_hybrid_topk_bf16. */
int cbrs_score_hybrid_topk_bf16_ex(const float *P1, const float *Q1, const float *P2, const float *Q2, int64_t n_users,
                                   int32_t n_items, int32_t c, const float *w3a2, const float *b3a2, const float *w3b2,
                                   const float *b3b2, const float *wc1, const float *bc1, const float *wc2,
                                   const float *bc2, const float *wc3, const float *bc3, int32_t k, int32_t *ids_out,
                                   float *scores_out, const int64_t *excl_rowptr, const int32_t *excl_items,
                                   void *workspace, size_t workspace_bytes, void *stream);
/* The same scorer at fp32 accuracy (1e-5 on the scores): each of the five 64 x 64 products runs as 3xTF32 on the tensor
 * cores (as cbrs_score_catalog_topk_tf32x3), every activation that feeds one split into a tf32 part and its remainder;
 * bias, relu, the output dot and the sigmoid in fp32.  Arguments and outputs as cbrs_score_hybrid_topk_bf16_ex, with
 * k in [1, min(128, n_items)]; slots past a user's eligible items hold -1 / -inf.  Exclusion lists as above
 * cbrs_score_catalog_topk_ex (both null: none; exactly one null: CBRS_E_INVALID).  c != 64: CBRS_E_UNSUPPORTED;
 * workspace: at least cbrs_score_hybrid_topk_tf32x3_workspace_bytes(), 16-byte aligned, else CBRS_E_WORKSPACE;
 * n_users == 0 writes nothing.                                                                                    */
size_t cbrs_score_hybrid_topk_tf32x3_workspace_bytes(void);
int cbrs_score_hybrid_topk_tf32x3(const float *P1, const float *Q1, const float *P2, const float *Q2, int64_t n_users,
                                  int32_t n_items, int32_t c, const float *w3a2, const float *b3a2, const float *w3b2,
                                  const float *b3b2, const float *wc1, const float *bc1, const float *wc2,
                                  const float *bc2, const float *wc3, const float *bc3, int32_t k, int32_t *ids_out,
                                  float *scores_out, const int64_t *excl_rowptr, const int32_t *excl_items,
                                  void *workspace, size_t workspace_bytes, void *stream);

/* Grouped transform of the relational layer (row R: "R-GCN per-relation transform plus scatter as a grouped kernel"):
 * ONE launch computes X[m, f] . [W_0 | ... | W_{R-1}] (w_cat: contiguous [f, n_groups*h], Keras layout) and stores
 * column block r of row m at row r*group_rows + m of `out` ([n_groups*group_rows, h], leading dimension ldo), i.e.
 * straight into the stacked operand whose column ids r*N + j the relational CSR (cbrs_graph_build_csr_rel) gathers
 * from - the sparse kernel that follows is the grouped scatter.  out_dtype / peers as cbrs_dense_ex.  The reference has
 * no relational layer (it drops the predicate column, src/data/loaders.py:63-68); n_groups = 1 is cbrs_dense.      */
int cbrs_dense_grouped(const float *x, int64_t ldx, const float *w_cat, int64_t m, int32_t f, int32_t h,
                       int32_t n_groups, void *out, int64_t ldo, int64_t group_rows, int out_dtype,
                       void *const *out_peers_host, int n_peers, void *stream);

/* fp32-ACCURATE Dense layer on the tensor cores: the GCN transform Z = X W (src/models/gnn.py:285-295: GCNConv =
 * transform, then propagate) at scaled-graph size.  out = act(X @ W + b), everything fp32; the product is split
 * into three kind::tf32 tcgen05 MMAs (Xl Wh + Xh Wl + Xh Wh with xh = tf32(x), xl = x - xh) accumulated in fp32 in
 * TMEM, which agrees with the fp32 FFMA kernel to ~1e-6 of the output scale (parity test: 1e-5 vs float64).
 * X tiles arrive by TMA (cp.async.bulk.tensor, SWIZZLE_128B); W is handed over as the operand image written by
 * cbrs_dense_tf32x3_prepare (cbrs_dense_tf32x3_image_bytes(k, n) bytes, 16-byte aligned; rewrite it when W changes).
 * Shapes: k % 32 == 0, n % 16 == 0, 16 <= n <= 256, both operand images resident in shared memory (k*n <= 16384):
 * cbrs_dense_tf32x3_eligible.  Rows of x 16-byte aligned.  out_peers_host / n_peers as in cbrs_dense_bcast;
 * out_dtype = CBRS_DTYPE_BF16 stores the fp32 result rounded to bf16 (ldo in elements, % 16 == 0), as cbrs_dense_ex.
 * A row's result does not depend on its position in the 128-row tile => identical bits under any row partition.  */
int cbrs_dense_tf32x3_eligible(int32_t k, int32_t n);
size_t cbrs_dense_tf32x3_image_bytes(int32_t k, int32_t n);
int cbrs_dense_tf32x3_prepare(const float *w, int32_t k, int32_t n, void *image, void *stream);
int cbrs_dense_tf32x3(const float *x, int64_t ldx, const void *w_image, const float *b, int64_t m, int32_t k,
                      int32_t n, int act, void *out, int64_t ldo, int out_dtype, void *const *out_peers_host,
                      int n_peers, void *stream);

/* General form: out = act( rowop( x @ W + addend + b ) ).  addend: optional [m, n] fp32 matrix (ld_add in elements) added
 * to the product; rowop = CBRS_ROWOP_NONE or CBRS_ROWOP_L2NORM.  GraphSageConv's dense part
 * relu(l2_normalize([x || agg] @ K + b)) (spektral GraphSageConv.call, built at src/models/gnn.py:354-361) runs as two such
 * products, x @ K[:f] and then agg @ K[f:] + the first + b (the two operand images of a 2f-deep kernel do not fit shared
 * memory at once).                                                                                                   */
int cbrs_dense_tf32x3_ex(const float *x, int64_t ldx, const void *w_image, const float *b, const float *addend,
                         int64_t ld_add, int rowop, int64_t m, int32_t k, int32_t n, int act, void *out, int64_t ldo,
                         int out_dtype, void *const *out_peers_host, int n_peers, void *stream);

/* The GAT transform on the same kernel (spektral GATConv built at src/models/gnn.py:321-328: z = x W, then the two
 * attention logits per node): out = X W (fp32) plus p[m] = out[m,:] . a_self and q[m] = out[m,:] . a_neigh, i.e.
 * cbrs_dense with CBRS_ROWOP_ATTN on the tensor cores.  q_peers_host as in cbrs_dense_bcast.                          */
int cbrs_dense_tf32x3_attn(const float *x, int64_t ldx, const void *w_image, int64_t m, int32_t k, int32_t n,
                           const float *a_self, const float *a_neigh, float *p_out, float *q_out, float *out,
                           int64_t ldo, void *const *out_peers_host, void *const *q_peers_host, int n_peers,
                           void *stream);

/* General form of cbrs_dense: the output (and its peer copies) can be written as bf16 (out_dtype =
 * CBRS_DTYPE_BF16, round to nearest even, ldo in elements) so that the GCN transform Z = X W feeds the bf16
 * sparse kernel without a conversion pass; out_peers_host / q_peers_host / n_peers as in cbrs_dense_bcast.  */
int cbrs_dense_ex(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2, int64_t ld2,
                  const int64_t *idx2, int32_t f2, const float *w, const float *b, int64_t m, int32_t n, int act,
                  int rowop, const float *a_self, const float *a_neigh, float *p_out, float *q_out, void *out,
                  int64_t ldo, int out_dtype, void *const *out_peers_host, void *const *q_peers_host, int n_peers,
                  void *stream);

/* ---- reduction of layer outputs (row P5) ------------------------------------
 * out = sum_l coef[l] * h_l  ('sum': 1, 'mean': add then divide by L, 'w-sum': w^2).
 * 'concatenation' and 'last' need no kernel.  src/layers/reduction.py:15-55.    */
int cbrs_reduce_layers(const float *const *h_host, const int64_t *ld_host, int32_t n_layers,
                       const float *coef_host, float divide_by, int64_t n_rows, int32_t d,
                       float *out, int64_t ldo, void *stream);

/* ---- row gather (row S1/S3 when a materialised batch is needed) ------------- */
int cbrs_gather_rows(const float *x, int64_t ldx, const int64_t *idx, int64_t m, int32_t d,
                     float *out, int64_t ldo, void *stream);

/* ---- per-user top-k (row T) ---------------------------------------------------
 * Catalog form: scores [n_users, n_items] row-major -> ids/vals [n_users, k],
 * descending score, ties to the LOWER item index (== stable sort of the
 * reference scorer's output).  k <= 128.                                        */
int cbrs_topk_rows(const float *scores, int64_t ld, int64_t n_users, int32_t n_items, int32_t k,
                   int32_t *ids_out, float *vals_out, void *stream);
/* Exclusion lists on a materialised score block (the generic catalog path): scores [n_rows, n_cols] (leading
 * dimension ld) holds catalog columns col_base .. col_base + n_cols - 1; every listed item of row r (contract above
 * cbrs_score_catalog_topk_ex) that falls in that range is overwritten with -inf.  Both lists null: nothing to do. */
int cbrs_exclude_cols(float *scores, int64_t ld, int64_t n_rows, int32_t n_cols, int32_t col_base,
                      const int64_t *excl_rowptr, const int32_t *excl_items, void *stream);
/* Pair-list form (src/utilities/metrics.py:21-34): stable sort by (user asc,
 * score desc), first k rows per user.  order_out [n_pairs] = input row of each
 * sorted position; rank_out [n_pairs] = position inside its user's run (keep rows
 * with rank < k).                                                               */
size_t cbrs_topk_pairs_workspace_bytes(int64_t n_pairs);
int cbrs_topk_pairs(const int64_t *users, const float *scores, int64_t n_pairs, int64_t n_users,
                    int32_t *order_out, int32_t *rank_out, void *workspace,
                    size_t workspace_bytes, void *stream);

/* ---- fused full-catalog scorer + top-k for the BasicRS classifier (rows S1/S2 + T) ---------
 * The caller hoists everything that depends on one entity (cbrs_dense):
 *   P[u,:] = unet(emb[u]) @ W1[:du] + b1  [n_users, c1]     Q[i,:] = inet(emb[i]) @ W1[du:]  [n_items, c1]
 * (W1 = first classifier kernel, src/models/basic.py:29,35-36).  Per pair the kernel evaluates
 *   sigmoid( relu( relu(P[u]+Q[i]) @ W2[c1,c2] + b2 ) . w3 + b3 )
 * and keeps each user's k best (score desc, lower item index on ties); the score matrix is
 * never written.  fp32 FFMA (parity 1e-5 with the reference scorer).  c1 % 4 == 0, c1 <= 256,
 * c2 <= 128, k <= 128.  ids_out / scores_out: [n_users, k], -1 / -inf past the catalog size. */
int cbrs_score_catalog_topk(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                            int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                            const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                            float *scores_out, void *stream);

/* ---- exclusion lists of the catalog scorers (the *_ex entry points and cbrs_exclude_cols) ----
 * Per scored user, catalog items that must not appear in its top-k (typically the items it rated in training).
 *   excl_rowptr int64 [n_users + 1]: absolute offsets into excl_items; row r's list is
 *   excl_items[excl_rowptr[r] .. excl_rowptr[r + 1]) (int32).  Row r is the r-th SCORED user (row r of P / of the
 *   score block), not a global user id: for the contiguous users u0.. pass excl_rowptr + u0, no copy needed.
 *   Items are catalog indices in [0, n_items) (item node id - n_users), the space ids_out uses; other values never match.
 *   Each list is sorted ascending; duplicates and empty rows are allowed.  An UNSORTED row may exclude any subset of its
 *   own items, and never causes a read outside [excl_rowptr[r], excl_rowptr[r + 1]).
 * Output form is unchanged (score desc, ties to the lower item index); slots past the number of eligible items hold
 * -1 / -inf.  Both pointers null: no lists, the same kernel bit for bit as the entry point without _ex; empty lists give
 * the same bits as no lists.  Exactly one of the two null: CBRS_E_INVALID.  Workspace sizes do not change.  The fused
 * kernels search a user's list only for a candidate that beats its current k-th score.                              */
int cbrs_score_catalog_topk_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                               int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                               const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                               const int64_t *excl_rowptr, const int32_t *excl_items, void *stream);

/* ---- full-catalog ranking metrics of top-k lists (binary relevance) -------------------------------------------------
 * ids [n_rows, k] int32, leading dimension ld >= k: row r is the top-k list of user users[r] (users null: user r), best
 * first, as the catalog scorers write it.  -1 marks an empty slot; no value outside [0, n_items) is ever a hit.
 * Relevance lists: rel_rowptr int64 [n_users + 1] / rel_items int32, the CSR form of the exclusion lists above, but rows
 * are GLOBAL user ids (row u = user u, whichever rows are scored).  Each row is sorted ascending, distinct, catalog
 * indices.  An unsorted or duplicated row may lose hits (a duplicate also counts in R_u); it never causes a read
 * outside [rel_rowptr[u], rel_rowptr[u + 1]).  A user outside [0, n_users), or both pointers null, has no relevant
 * items.  Exactly one of the two pointers null: CBRS_E_INVALID.
 * cutoffs_host: n_cutoffs (1..8) strictly ascending cutoffs c in [1, k], host memory; k <= 128.
 * Per scored user with R_u = |rel_u| >= 1, hit_r = (slot r is in rel_u), at each cutoff c:
 *   P = sum_{r<c} hit_r / c            R = sum_{r<c} hit_r / R_u            HR = 1 if any hit_r with r < c
 *   MRR = 1 / (r + 1) of the first hit at r < c, else 0
 *   NDCG = DCG / IDCG, DCG = sum_{r<c} hit_r / log2(r + 2), IDCG = sum_{r<min(c, R_u)} 1 / log2(r + 2)
 *   AP = sum_{r<c} hit_r * (sum_{s<=r} hit_s) / (r + 1) / min(c, R_u)
 * sums_out fp64 [n_cutoffs, 7] (device): columns P, R, HR, MRR, NDCG, AP summed over the scored users with R_u >= 1,
 * and column 6 the number of those users.  Rows without relevant items add nothing.  The sums are bit-identical from
 * run to run and do not depend on ld: the rows are added in a fixed tree over fixed blocks of rows.
 * per_user_out fp64 [n_rows, n_cutoffs, 6] (may be null): the six values of row r; NaN for a row with R_u = 0.
 * Workspace: cbrs_rank_metrics_workspace_bytes(n_rows, n_cutoffs) bytes, 8-byte aligned, else CBRS_E_WORKSPACE.
 * Every argument is checked before any launch.                                                                      */
size_t cbrs_rank_metrics_workspace_bytes(int64_t n_rows, int32_t n_cutoffs);
int cbrs_rank_metrics(const int32_t *ids, int64_t ld, int64_t n_rows, int32_t k, int32_t n_items, const int64_t *users,
                      int64_t n_users, const int64_t *rel_rowptr, const int32_t *rel_items, const int32_t *cutoffs_host,
                      int32_t n_cutoffs, double *sums_out, double *per_user_out, void *workspace,
                      size_t workspace_bytes, void *stream);

/* The same scorer with the 64 x 64 product on the tensor cores at fp32 accuracy (3xTF32: h = relu(P[u]+Q[i]) and W2 are
 * split into a tf32 part and an exact remainder, three kind::tf32 MMAs per K step accumulate in fp32; the A operand is
 * written by its threads straight into tensor memory).  Same contract, outputs and tie rule as cbrs_score_catalog_topk;
 * scores agree with it to ~1e-6 (1e-5 stated in the tests).  Shapes: c1 in {32, 64}, c2 <= 64 (the reference's grids:
 * clf_units [64, 64]); anything else: cbrs_score_catalog_topk.  Workspace: the operand images of W2.            */
int cbrs_score_catalog_topk_tf32x3_eligible(int32_t c1, int32_t c2);
size_t cbrs_score_catalog_topk_tf32x3_workspace_bytes(int32_t c1, int32_t c2);
int cbrs_score_catalog_topk_tf32x3(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                   int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                   const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                                   float *scores_out, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_score_catalog_topk_tf32x3_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                      int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                      const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                                      const int64_t *excl_rowptr, const int32_t *excl_items, void *workspace,
                                      size_t workspace_bytes, void *stream);

/* bf16 tensor-core variant (tcgen05.mma, TMEM accumulator): same contract and arguments; the
 * per-pair activations relu(P[u]+Q[i]) and W2 are rounded to bf16, accumulation is fp32, so
 * scores differ from the fp32 kernel by O(1e-3) (tolerance stated in tests).  c1 % 8 == 0,
 * c1 <= 256, c2 <= 256.  For c1 <= 64 (the reference's grids) P and Q themselves are rounded to bf16 and
 * added with add.rn.bf16x2: h1 = bf16(bf16(P) + bf16(Q)); for wider c1 the sum is formed in fp32 and
 * rounded once.  Workspace: the pre-swizzled bf16 image of W2^T (+ Q as bf16 when c1 <= 64).              */
size_t cbrs_score_catalog_topk_bf16_workspace_bytes(int32_t n_items, int32_t c1, int32_t c2);
int cbrs_score_catalog_topk_bf16(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                 int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                 const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                                 float *scores_out, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_score_catalog_topk_bf16_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                    int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                    const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                                    const int64_t *excl_rowptr, const int32_t *excl_items, void *workspace,
                                    size_t workspace_bytes, void *stream);

/* ---- synthetic scaled graph (SURVEY 8d, config 5) --------------------------------
 * Counter-based generator: edge e connects user hash_u(seed,e) % n_users with an
 * item drawn from a capped Zipf(1) popularity; writes BOTH directions, i.e.
 * 2*n_edges COO entries: (u, U+i) for e < n_edges then (U+i, u).                */
int cbrs_synth_bipartite(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed,
                         int32_t *coo_row, int32_t *coo_col, void *stream);
/* scatter_items = 0: item id = popularity rank (no multiplicative scattering), i.e. ids as np.unique would leave a
 * catalogue that is sorted by popularity - the adversarial case for a row-count partition (SURVEY 8e).  1 = as above. */
int cbrs_synth_bipartite_ex(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed, int scatter_items,
                            int32_t *coo_row, int32_t *coo_col, void *stream);
/* The entries of edges [edge_lo, edge_hi) only, 2*(edge_hi - edge_lo) of them: the forward entries of those edges
 * in [0, m) and their reverses in [m, 2m), m = edge_hi - edge_lo, each with the bits cbrs_synth_bipartite_ex writes
 * for that edge.  The forward parts of consecutive ranges, then their reverse parts, make up the whole output:
 * a graph can be streamed in fixed-size pieces instead of holding all 2*n_edges entries.                          */
int cbrs_synth_bipartite_range(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed, int scatter_items,
                               int64_t edge_lo, int64_t edge_hi, int32_t *coo_row, int32_t *coo_col, void *stream);

/* ---- peer memory + producer kernels that store into every rank's copy (SURVEY 8e; multi-GPU) ---
 * One process per GPU.  Every rank allocates the same ("symmetric") buffers with
 * cbrs_peer_alloc, exports an IPC handle (CBRS_IPC_HANDLE_BYTES opaque bytes, exchanged by
 * the host, e.g. torch.distributed.all_gather_object) and maps its peers' copies with
 * cbrs_peer_open.  The *_bcast kernels store every finished output row into the local
 * buffer AND into the n_peers peer-mapped copies (same layout; plain stores over
 * NVLink/NVSwitch), so the all-gather of a layer's operand happens inside the kernel that
 * produces it.  cbrs_peer_barrier is the stream-ordered rendezvous that follows: rank r
 * publishes `epoch` (monotonically increasing, same on all ranks) into slot r of every
 * rank's flag array and waits until all slots of its own array reach `epoch`; *status
 * (device int32, zeroed by the caller) becomes 1 if a peer did not arrive within
 * timeout_s AND the kernel traps: the consumers would otherwise gather from partly written
 * operand buffers, so the stream fails (every later CUDA call of the process returns an
 * error) instead of continuing.  The reference has no multi-device code; these calls replace the
 * all-gather + barrier a NCCL-based port would issue per layer.                           */
#define CBRS_MAX_PEERS 8
#define CBRS_IPC_HANDLE_BYTES 64
int cbrs_peer_alloc(size_t bytes, void **ptr_out); /* cudaMalloc'd (IPC-exportable), zero-filled */
int cbrs_peer_free(void *ptr);
int cbrs_peer_export(void *ptr, unsigned char *handle_host);
int cbrs_peer_open(const unsigned char *handle_host, void **ptr_out);
int cbrs_peer_close(void *ptr);

/* Coalesced copy of a row block (m rows of w floats, leading dimensions in elements) into a MAPPED address: the same view
 * in a peer's copy of a symmetric buffer, or in the buffer's NVSwitch multicast mapping (one store reaches every copy).
 * Used where the producing kernel's own stores would reach the fabric as scattered 32-byte pieces (the epilogues of the
 * tensor-core Dense kernels write one row per thread): the kernel stores locally, this pushes the finished block.     */
int cbrs_push_rows(const float *src, int64_t lds, void *dst, int64_t ldd, int64_t m, int32_t w, void *stream);
/* flags_peers_host[r] = rank r's flag array (uint64[CBRS_MAX_PEERS], peer-mapped; own for r == my_rank) */
int cbrs_peer_barrier(void *const *flags_peers_host, int n_ranks, int my_rank, uint64_t epoch,
                      int32_t *status, double timeout_s, void *stream);
/* cbrs_spmm_csr + stores into y_peers_host[0..n_peers) (each the peer's address of the same y view) */
int cbrs_spmm_csr_bcast(const cbrs_csr_t *g, const void *x, int64_t ldx, void *y, int64_t ldy, int32_t d,
                        int agg, const float *bias, int relu, int dtype, void *const *y_peers_host,
                        int n_peers, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_gat_csr_bcast(const cbrs_csr_t *g, int64_t row_offset, const float *z, int64_t ldz, const float *p,
                       const float *q, float *y, int64_t ldy, int32_t h, const float *bias, int relu,
                       void *const *y_peers_host, int n_peers, void *workspace, size_t workspace_bytes,
                       void *stream);
/* cbrs_dense + stores of out (and q for the attention row-op) into the peers' copies */
int cbrs_dense_bcast(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2,
                     int64_t ld2, const int64_t *idx2, int32_t f2, const float *w, const float *b, int64_t m,
                     int32_t n, int act, int rowop, const float *a_self, const float *a_neigh, float *p_out,
                     float *q_out, float *out, int64_t ldo, void *const *out_peers_host,
                     void *const *q_peers_host, int n_peers, void *stream);

/* ---- id compaction (rows G0 / (f)-2) ------------------------------------------------------------
 * cbrs_compact_ids == np.unique(ids, return_inverse=True) (src/data/loaders.py:47-49,65): uniques_out
 * (capacity n) receives the sorted distinct values, inverse_out[i] the index of ids[i] among them,
 * *n_unique_out (device) their count.  cbrs_lookup_ids replaces the `col[:,None] == vocab` broadcast +
 * argwhere of loaders.py:53-54,64 with a binary search; ids absent from the vocabulary give -1 (the
 * reference silently drops such rows; the host wrapper raises).  Bit-exact integer work.             */
size_t cbrs_compact_ids_workspace_bytes(int64_t n);
int cbrs_compact_ids(const int64_t *ids, int64_t n, int64_t *uniques_out, int64_t *inverse_out,
                     int64_t *n_unique_out, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_lookup_ids(const int64_t *vocab_sorted, int64_t n_vocab, const int64_t *ids, int64_t n,
                    int64_t *index_out, void *stream);

/* ---- DGCF operator build and layer pieces (scope row (f)-3) -------------------------------------
 * Replaces, on device, DGCFConv.preprocess / high_pass_filter (src/layers/dgcf_conv.py:38-80; scipy on
 * the host in the reference) and LocalityAdaptive.call (:101-102).
 * A.dot(A) -> cbrs_spgemm_count (row_offsets [n_rows] = exclusive scan of the products per row,
 * *total_out device int64) + cbrs_spgemm_expand (COO of the elementary products a_ik*a_kj, row-major,
 * k ascending) -> cbrs_graph_build_csr sums the duplicates (and applies gcn_filter).                 */
size_t cbrs_spgemm_workspace_bytes(int64_t n_rows);
int cbrs_spgemm_count(const cbrs_csr_t *left, const cbrs_csr_t *right, int64_t *row_offsets, int64_t *total_out,
                      void *workspace, size_t workspace_bytes, void *stream);
int cbrs_spgemm_expand(const cbrs_csr_t *left, const cbrs_csr_t *right, const int64_t *row_offsets,
                       int32_t *coo_row, int32_t *coo_col, float *coo_val, void *stream);
/* counts[j] (device uint64) = #{i : vals[i] > eps_host[j]}, j < n_eps <= 8: the threshold search of
 * high_pass_filter (dgcf_conv.py:60-80) */
int cbrs_count_above(const float *vals, int64_t n, const float *eps_host, int32_t n_eps, uint64_t *counts,
                     void *stream);
/* COO (row-major order kept) of the CSR entries with value > eps; capacity = the count from cbrs_count_above */
size_t cbrs_csr_filter_above_workspace_bytes(int64_t nnz);
int cbrs_csr_filter_above(const cbrs_csr_t *g, float eps, int32_t *coo_row, int32_t *coo_col, float *coo_val,
                          void *workspace, size_t workspace_bytes, void *stream);
/* LocalityAdaptive: out[r,:] = x[r,:] * sigmoid(w[r]); backward: dx = g*sigmoid(w), dw[r] = sigmoid'(w[r]) * g[r,:].x[r,:] */
int cbrs_row_gate(const float *x, int64_t ldx, const float *w, int64_t rows, int32_t d, float *out, int64_t ldo,
                  void *stream);
int cbrs_row_gate_grad(const float *g, int64_t ldg, const float *x, int64_t ldx, const float *w, int64_t rows,
                       int32_t d, float *dx, int64_t lddx, float *dw, void *stream);

/* ---- training step (scope row (f)-1) ------------------------------------------------------
 * The reference differentiates with TensorFlow autograd inside Keras `fit`
 * (src/experiment.py:155-188): loss = binary cross-entropy (config.yaml:50) + l2 * sum w^2 over
 * the embeddings and GNN kernels/biases (src/models/gnn.py:239-246), optimiser Adam(1e-3, 0.9)
 * (config.yaml:52-56).  Here each derivative is an explicit kernel; the sparse backward is
 * cbrs_spmm_csr itself (A_hat is symmetric) and dX = dPre W^T is cbrs_dense on W^T.
 * All reductions use a fixed order: gradients are reproducible run to run.                  */
/* dPre = dOut * act'(out) for CBRS_ACT_*; 2-D strided views */
int cbrs_act_grad(const float *dout, int64_t ldd, const float *out, int64_t ldo, int64_t rows, int32_t d,
                  int act, float *dpre, int64_t ldp, void *stream);
/* dW[f1+f2, n] = [X1[idx1] || X2[idx2]]^T dPre[m, n];  db[n] = column sums of dPre (db may be NULL) */
size_t cbrs_dense_grad_w_workspace_bytes(int64_t m, int32_t k, int32_t n);
int cbrs_dense_grad_w(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2,
                      int64_t ld2, const int64_t *idx2, int32_t f2, const float *dpre, int64_t ldd, int64_t m,
                      int32_t n, float *dw, float *db, void *workspace, size_t workspace_bytes, void *stream);
int cbrs_transpose_f32(const float *src, int32_t rows, int32_t cols, float *dst, void *stream);
/* dst[idx[m], 0:d] += src[m, 0:d]  (backward of tf.nn.embedding_lookup, src/models/basic.py:72-75);
 * duplicates are added in ascending m */
size_t cbrs_scatter_add_rows_workspace_bytes(int64_t m);
int cbrs_scatter_add_rows(const float *src, int64_t lds, const int64_t *idx, int64_t m, int32_t d,
                          int64_t n_rows, float *dst, int64_t ldd, void *workspace, size_t workspace_bytes,
                          void *stream);
/* GraphSageConv epilogue as its own kernel (training keeps the pre-normalisation v) and its backward */
int cbrs_l2norm_act(const float *v, int64_t ldv, int64_t rows, int32_t d, int relu, float *out, int64_t ldo,
                    void *stream);
int cbrs_l2norm_relu_grad(const float *v, int64_t ldv, const float *dout, int64_t ldd, int64_t rows, int32_t d,
                          int relu, float *dv, int64_t ldo, void *stream);
/* out[r,:] = x[r,:] / (rowptr[r+1]-rowptr[r])  (0 for empty rows): mean-aggregator backward = A^T (dAgg / deg) */
int cbrs_scale_rows_inv_degree(const float *x, int64_t ldx, const int64_t *rowptr, int64_t rows, int32_t d,
                               float *out, int64_t ldo, void *stream);
/* out = ca*a + cb*b (b may be NULL) on strided 2-D views */
int cbrs_axpby2d(const float *a, int64_t lda, float ca, const float *b, int64_t ldb, float cb, int64_t rows,
                 int32_t d, float *out, int64_t ldo, void *stream);
/* Keras binary_crossentropy on probabilities (clipped to [1e-7, 1-1e-7]): *loss_out = mean; dp_out[i] =
 * dLoss/dp_i (0 where the clip is active); *correct_out = #((p > .5) == (y > .5)).  dp/correct may be NULL */
int cbrs_bce(const float *p, const float *y, int64_t n, float *loss_out, float *dp_out, float *correct_out,
             void *stream);
/* *out = (accumulate ? *out : 0) + scale * sum w^2; two-level fixed-order reduction (reproducible) */
size_t cbrs_sum_squares_workspace_bytes(void);
int cbrs_sum_squares(const float *w, int64_t n, float scale, float *out, int accumulate, void *workspace,
                     size_t workspace_bytes, void *stream);
/* Keras Adam: g' = g + 2*l2*w; m,v updated in place; w -= lr_t * m / (sqrt(v) + eps).  lr_t = lr*sqrt(1-b2^t)/(1-b1^t)
 * is computed by the host; lr_t_dev (device float, may be NULL) overrides the immediate so that a captured
 * CUDA graph of the whole step can be replayed with the rate of step t                                        */
int cbrs_adam_step(float *w, const float *g, float *m, float *v, int64_t n, float lr_t, const float *lr_t_dev,
                   float beta1, float beta2, float eps, float l2, void *stream);

/* Hybrid tweaks grid (scope row (f)-3).  FusionLayer('attention') (src/layers/fusion.py:56-68) with
 * ta = tanh(a W), tb = tanh(b W) from two cbrs_dense calls: out = softmax2(ta, tb) . (a, b) per feature; ta/tb/da/
 * db/dta/dtb are contiguous [rows, d].  cbrs_add3_act: activation(residual(x) + x1 + x2) (src/models/hybrid.py:89). */
int cbrs_attn_fuse(const float *a, int64_t lda, const float *b, int64_t ldb, const float *ta, const float *tb,
                   int64_t rows, int32_t d, float *out, int64_t ldo, void *stream);
int cbrs_attn_fuse_grad(const float *g, int64_t ldg, const float *a, int64_t lda, const float *b, int64_t ldb,
                        const float *ta, const float *tb, int64_t rows, int32_t d, float *da, float *db,
                        float *dta, float *dtb, void *stream);
int cbrs_add3_act(const float *a, int64_t lda, const float *b, int64_t ldb, const float *c, int64_t ldc,
                  int64_t rows, int32_t d, int act, float *out, int64_t ldo, void *stream);
/* Backward of cbrs_gat_csr (fused edge-softmax gradient).  d_o = dY * act'(y).  Outputs: dz [N,h] =
 * sum_i alpha_ij dO_i + dp (x) a_self + dq (x) a_neigh (the full gradient w.r.t. z = X W), dp, dq [N] (for
 * d a_self = z^T dp, d a_neigh = z^T dq).  The graph must be structurally symmetric (every adjacency of the
 * reference is, config.yaml:36): the edges ending in a node are read from that node's own row.  Full graph
 * only (g->n_rows == N); rows are not chunked (training runs at MovieLens scale).                        */
size_t cbrs_gat_backward_workspace_bytes(int64_t n_rows);
int cbrs_gat_backward(const cbrs_csr_t *g, const float *z, int64_t ldz, const float *p, const float *q,
                      const float *y, int64_t ldy, const float *bias, const float *d_o, int64_t ldo, int32_t h,
                      const float *a_self, const float *a_neigh, float *dz, int64_t lddz, float *dp, float *dq,
                      void *workspace, size_t workspace_bytes, void *stream);
/* cbrs_gat_backward on rows [row_offset, row_offset + g->n_rows) of the graph (a row slice with global column ids,
 * as cbrs_gat_csr takes), in two phases so that an exchange can sit between them under a row partition:
 *   stats_rows: (m_i, S_i, t_i) of the slice's rows into `stats` (the slice's rows of an [N, 3] contiguous array) and
 *               into stats_peers_host[0..n_peers) (each a peer's address of the same view);
 *   grad_rows:  dz, dp, dq of the slice's rows, the combine included, into dz/dp/dq and the peers' copies.  `stats` is
 *               the whole [N, 3] array: the phase reads the stats of every neighbour row, so all rows' stats must be
 *               there first.
 * Inputs p, q, y, d_o and z are whole-graph arrays ([N] / [N, ld]) read at global rows; outputs are views of the
 * slice's rows, as cbrs_gat_csr's y.  Each output row has the bits the whole-graph call gives it.  For an NVSwitch multicast target pass the multicast address of the output as the output and n_peers = 0: no
 * kernel reads its outputs back.  Null arguments, a null peer copy, n_peers > CBRS_MAX_PEERS - 1, h > 256 and a bad
 * leading dimension or row_offset return CBRS_E_INVALID before any launch.  No workspace.                       */
int cbrs_gat_backward_stats_rows(const cbrs_csr_t *g, int64_t row_offset, const float *p, const float *q,
                                 const float *y, int64_t ldy, const float *bias, const float *d_o, int64_t ldo,
                                 int32_t h, float *stats, void *const *stats_peers_host, int n_peers, void *stream);
int cbrs_gat_backward_grad_rows(const cbrs_csr_t *g, int64_t row_offset, const float *z, int64_t ldz, const float *p,
                                const float *q, const float *d_o, int64_t ldo, int32_t h, const float *stats,
                                const float *a_self, const float *a_neigh, float *dz, int64_t lddz, float *dp,
                                float *dq, void *const *dz_peers_host, void *const *dp_peers_host,
                                void *const *dq_peers_host, int n_peers, void *stream);
/* the same update for all n_tensors weight tensors of a model in one launch (host arrays of device pointers) */
int cbrs_adam_step_multi(int32_t n_tensors, void *const *w_host, const void *const *g_host, void *const *m_host,
                         void *const *v_host, const int64_t *n_host, const float *l2_host, float lr_t,
                         const float *lr_t_dev, float beta1, float beta2, float eps, void *stream);

/* ---- primitives exported for tests -------------------------------------------- */
size_t cbrs_sort_workspace_bytes(int64_t n);
/* stable ascending sort of 64-bit keys (bits [0,key_bits)) with a 32-bit payload */
int cbrs_sort_pairs_u64(uint64_t *keys, uint32_t *payload, int64_t n, int key_bits,
                        void *workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CBRS_B200_H_ */
