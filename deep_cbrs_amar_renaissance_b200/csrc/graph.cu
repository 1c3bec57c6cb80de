// Device graph build: COO -> (row,[rel,]col)-sorted CSR, duplicate sum, self loops,
// symmetric normalisation, and the chunk decomposition used by the propagation
// kernels.  Rows G1-G3 of SURVEY.md section 8a.
//
// What it replaces: scipy's coo->csr (+sum_duplicates) and spektral.utils.gcn_filter
// at /root/reference/src/models/gnn.py:283, src/layers/lightgcn_conv.py:58, and the
// tf.sparse.reorder of src/utilities/math.py:47-56.  All integer outputs are
// bit-exact against the oracle (oracle/graph.py); values are exact for the 0/1
// adjacencies the reference builds (d = fl32(1/sqrt(double(deg)))).
#include "common.cuh"

namespace cbrs {

constexpr int kThreads = 256;

static int bits_for(int64_t n) {  // bits needed to hold values in [0, n)
    int b = 1;
    while (((int64_t)1 << b) < n) ++b;
    return b;
}

struct KeyLayout {
    int col_bits, rel_bits, row_bits;
    __host__ __device__ int key_bits() const { return col_bits + rel_bits + row_bits + 1; }  // +1: invalid flag on top
    __host__ __device__ uint64_t invalid() const { return 1ull << (col_bits + rel_bits + row_bits); }
    __device__ uint64_t pack(int64_t r, int64_t rel, int64_t c) const {
        return ((uint64_t)r << (col_bits + rel_bits)) | ((uint64_t)rel << col_bits) | (uint64_t)c;
    }
    __device__ int64_t row(uint64_t k) const { return (int64_t)(k >> (col_bits + rel_bits)); }
    __device__ int64_t rel(uint64_t k) const { return (int64_t)((k >> col_bits) & ((1ull << rel_bits) - 1)); }
    __device__ int64_t col(uint64_t k) const { return (int64_t)(k & ((1ull << col_bits) - 1)); }
};

// Rows [row_lo, row_lo + n_rows) of an n_cols-node graph (the whole build: row_lo = 0, n_rows = n_cols); keys carry
// the row relative to row_lo, entries of other rows are invalid.
__global__ void make_keys_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                 const int32_t *__restrict__ rel, const float *__restrict__ val, int64_t nnz,
                                 int64_t row_lo, int64_t n_rows, int64_t n_cols, int64_t n_loops, int32_t self_rel,
                                 int drop_diag, KeyLayout kl, uint64_t *__restrict__ keys, uint32_t *__restrict__ payload) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz + n_loops) return;
    if (i < nnz) {
        const int64_t r = (int64_t)row[i] - row_lo, c = col[i];
        const bool bad = r < 0 || c < 0 || r >= n_rows || c >= n_cols || (drop_diag && r + row_lo == c);
        keys[i] = bad ? kl.invalid() : kl.pack(r, rel ? rel[i] : 0, c);
        payload[i] = val ? __float_as_uint(val[i]) : __float_as_uint(1.0f);
    } else {  // appended diagonal: M_ii += 1 falls out of the duplicate sum
        const int64_t d = i - nnz;
        keys[i] = kl.pack(d, self_rel, row_lo + d);
        payload[i] = __float_as_uint(1.0f);
    }
}

__device__ __forceinline__ bool is_head(const uint64_t *keys, int64_t i, uint64_t invalid, int dedup) {
    const uint64_t k = keys[i];
    if (k >= invalid) return false;
    if (!dedup || i == 0) return true;
    return keys[i - 1] != k;
}

__global__ void head_flags_kernel(const uint64_t *__restrict__ keys, int64_t n, uint64_t invalid, int dedup,
                                  uint32_t *__restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = is_head(keys, i, invalid, dedup) ? 1u : 0u;
}

// One thread per sorted input entry.  Heads write their compacted edge (summing their run
// in sorted == input order); row boundaries fill the row-pointer gaps.
__global__ void compact_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ payload,
                               const uint32_t *__restrict__ pos, const uint32_t *__restrict__ total, int64_t n,
                               int64_t n_rows, int64_t n_cols, KeyLayout kl, int dedup, int64_t *__restrict__ rowptr,
                               int32_t *__restrict__ colidx, float *__restrict__ vals, int64_t *__restrict__ nnz_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && nnz_out) *nnz_out = (int64_t)*total;
    if (i >= n) return;
    const uint64_t inv = kl.invalid();
    const uint64_t k = keys[i];
    if (k >= inv) return;
    const int64_t r = kl.row(k);
    const bool head = !dedup || i == 0 || keys[i - 1] != k;
    if (head) {
        const uint32_t o = pos[i];
        colidx[o] = (int32_t)(kl.rel(k) * n_cols + kl.col(k));
        float acc = __uint_as_float(payload[i]);
        if (dedup)
            for (int64_t j = i + 1; j < n && keys[j] == k; ++j) acc += __uint_as_float(payload[j]);
        vals[o] = acc;
        const int64_t prev_row = (i == 0) ? -1 : kl.row(keys[i - 1]);
        for (int64_t rr = prev_row + 1; rr <= r; ++rr) rowptr[rr] = (int64_t)o;  // empty rows share the offset
    }
    const bool last_valid = (i + 1 == n) || keys[i + 1] >= inv;
    if (last_valid) {
        const int64_t t = (int64_t)*total;
        for (int64_t rr = r + 1; rr <= n_rows; ++rr) rowptr[rr] = t;
    }
}

// warp per row: row sum with a fixed shuffle tree, then d = fl32(1/sqrt(double(sum)))
__global__ void __launch_bounds__(kThreads) inv_sqrt_degree_kernel(const int64_t *__restrict__ rowptr,
                                                                   const float *__restrict__ vals, int64_t n_rows,
                                                                   float *__restrict__ dinv) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    float s = 0.f;
    for (int64_t j = b + lane; j < e; j += 32) s += vals[j];
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        const double d = 1.0 / sqrt((double)s);
        const float f = (float)d;
        dinv[row] = isinf(f) ? 0.f : f;
    }
}

// d_i from dinv_rows[row] (the rows held here), d_j from dinv[column] (every node)
__global__ void __launch_bounds__(kThreads) sym_scale_kernel(const int64_t *__restrict__ rowptr,
                                                             const int32_t *__restrict__ colidx,
                                                             const float *__restrict__ dinv_rows,
                                                             const float *__restrict__ dinv, int64_t n_rows,
                                                             int64_t n_nodes, float *__restrict__ vals) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    const float di = dinv_rows[row];
    for (int64_t j = b + lane; j < e; j += 32) {
        const int64_t c = (int64_t)colidx[j] % n_nodes;  // strip the relation block
        vals[j] = __fmul_rn(__fmul_rn(di, vals[j]), dinv[c]);
    }
}

static size_t graph_ws_bytes(int64_t nnz, int64_t n_nodes, int flags) {
    const int64_t n_in = nnz + ((flags & CBRS_GRAPH_ADD_SELF_LOOPS) ? n_nodes : 0);
    return align_up((size_t)n_in * 8) + align_up((size_t)n_in * 4) + align_up((size_t)n_in * 4) + 256 /*total*/ +
           align_up((size_t)n_nodes * 4) +
           (sort_workspace_bytes(n_in) > scan_u32_workspace_bytes(n_in) ? sort_workspace_bytes(n_in)
                                                                        : scan_u32_workspace_bytes(n_in)) +
           4096;
}

// Rows [row_lo, row_lo + n_rows) of the n_nodes-node graph (the whole graph: row_lo = 0, n_rows = n_nodes).  With
// SYM_NORM: dinv_out == NULL scales the values here (the rows' own d serves every column: the whole graph only);
// otherwise the rows' d goes to dinv_out and the values stay unscaled (cbrs_graph_block_scale finishes them).
static int build(const int32_t *coo_row, const int32_t *coo_col, const int32_t *coo_rel, const float *coo_val,
                 int64_t nnz, int64_t row_lo, int64_t n_rows, int64_t n_nodes, int32_t n_rel, int32_t self_rel,
                 int flags, int64_t *rowptr, int32_t *colidx, float *vals, float *dinv_out, int64_t *nnz_out, void *ws,
                 size_t ws_bytes, cudaStream_t s) {
    CBRS_REQUIRE(nnz >= 0 && n_nodes > 0 && n_rel >= 1, CBRS_E_INVALID, "graph_build: nnz=%lld n=%lld n_rel=%d",
                 (long long)nnz, (long long)n_nodes, n_rel);
    CBRS_REQUIRE(row_lo >= 0 && n_rows > 0 && row_lo + n_rows <= n_nodes, CBRS_E_INVALID,
                 "graph_build: rows [%lld, %lld) of %lld", (long long)row_lo, (long long)(row_lo + n_rows),
                 (long long)n_nodes);
    CBRS_REQUIRE(dinv_out || !(flags & CBRS_GRAPH_SYM_NORM) || (row_lo == 0 && n_rows == n_nodes), CBRS_E_INVALID,
                 "graph_build: a row block needs dinv_out for SYM_NORM");
    CBRS_REQUIRE(rowptr && colidx && vals, CBRS_E_INVALID, "graph_build: null output");
    CBRS_REQUIRE(nnz == 0 || (coo_row && coo_col), CBRS_E_INVALID, "graph_build: null input");
    CBRS_REQUIRE(!(flags & CBRS_GRAPH_ADD_SELF_LOOPS) || (flags & CBRS_GRAPH_DEDUP_SUM), CBRS_E_INVALID,
                 "graph_build: ADD_SELF_LOOPS requires DEDUP_SUM");
    CBRS_REQUIRE((int64_t)n_rel * n_nodes < ((int64_t)1 << 31), CBRS_E_INVALID, "graph_build: n_rel*n_nodes overflows int32");
    CBRS_REQUIRE(self_rel >= 0 && self_rel < n_rel, CBRS_E_INVALID, "graph_build: self_rel=%d", self_rel);
    const int64_t n_loops = (flags & CBRS_GRAPH_ADD_SELF_LOOPS) ? n_rows : 0;
    const int64_t n_in = nnz + n_loops;
    CBRS_REQUIRE(n_in < (int64_t)0xfffffff0ll, CBRS_E_INVALID, "graph_build: %lld entries exceed the 32-bit position range",
                 (long long)n_in);
    KeyLayout kl;
    kl.col_bits = bits_for(n_nodes);
    kl.row_bits = bits_for(n_rows);
    kl.rel_bits = n_rel > 1 ? bits_for(n_rel) : 0;
    CBRS_REQUIRE(kl.key_bits() <= 64, CBRS_E_INVALID, "graph_build: key needs %d bits", kl.key_bits());

    Arena a(ws, ws_bytes);
    uint64_t *keys = a.take<uint64_t>((size_t)n_in);
    uint32_t *payload = a.take<uint32_t>((size_t)n_in);
    uint32_t *pos = a.take<uint32_t>((size_t)n_in);
    uint32_t *total = a.take<uint32_t>(1);
    float *dinv = a.take<float>((size_t)n_rows);
    CBRS_REQUIRE(keys && payload && pos && total && dinv, CBRS_E_WORKSPACE, "graph_build: workspace too small");
    void *sub = (char *)ws + a.off;
    const size_t sub_bytes = ws_bytes - a.off;

    cudaMemsetAsync(rowptr, 0, (size_t)(n_rows + 1) * sizeof(int64_t), s);
    cudaMemsetAsync(total, 0, sizeof(uint32_t), s);
    if (nnz_out) cudaMemsetAsync(nnz_out, 0, sizeof(int64_t), s);
    if (n_in == 0) return CBRS_OK;
    const unsigned gb = (unsigned)cdiv(n_in, kThreads);
    make_keys_kernel<<<gb, kThreads, 0, s>>>(coo_row, coo_col, coo_rel, coo_val, nnz, row_lo, n_rows, n_nodes, n_loops,
                                             self_rel, (flags & CBRS_GRAPH_DROP_DIAG) ? 1 : 0, kl, keys, payload);
    CBRS_CHECK_LAUNCH("make_keys");
    int rc = sort_pairs_u64(keys, payload, n_in, kl.key_bits(), sub, sub_bytes, s);
    if (rc) return rc;
    const int dedup = (flags & CBRS_GRAPH_DEDUP_SUM) ? 1 : 0;
    head_flags_kernel<<<gb, kThreads, 0, s>>>(keys, n_in, kl.invalid(), dedup, pos);
    CBRS_CHECK_LAUNCH("head_flags");
    rc = scan_u32_exclusive(pos, n_in, total, sub, sub_bytes, s);
    if (rc) return rc;
    compact_kernel<<<gb, kThreads, 0, s>>>(keys, payload, pos, total, n_in, n_rows, n_nodes, kl, dedup, rowptr, colidx,
                                           vals, nnz_out);
    CBRS_CHECK_LAUNCH("compact");
    if (flags & CBRS_GRAPH_SYM_NORM) {
        const unsigned gr = (unsigned)cdiv(n_rows * 32, kThreads);
        inv_sqrt_degree_kernel<<<gr, kThreads, 0, s>>>(rowptr, vals, n_rows, dinv_out ? dinv_out : dinv);
        CBRS_CHECK_LAUNCH("inv_sqrt_degree");
        if (!dinv_out) {
            sym_scale_kernel<<<gr, kThreads, 0, s>>>(rowptr, colidx, dinv, dinv, n_rows, n_nodes, vals);
            CBRS_CHECK_LAUNCH("sym_scale");
        }
    }
    return CBRS_OK;
}

// ------------------------------------------------------------------ row selection (partitioned build)
__global__ void row_histogram_kernel(const int32_t *__restrict__ row, int64_t n, int64_t n_rows,
                                     unsigned long long *__restrict__ counts) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t r = row[i];
    if (r >= 0 && r < n_rows) atomicAdd(counts + r, 1ull);
}

__global__ void select_flags_kernel(const int32_t *__restrict__ row, int64_t n, int64_t lo, int64_t hi,
                                    uint32_t *__restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = (row[i] >= lo && row[i] < hi) ? 1u : 0u;
}

// pos = exclusive scan of the flags: entry i goes to *cursor + pos[i], i.e. selected entries keep their input order
__global__ void select_scatter_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                      const float *__restrict__ val, int64_t n, int64_t lo, int64_t hi, int rebase,
                                      const uint32_t *__restrict__ pos, const int64_t *__restrict__ cursor,
                                      int64_t capacity, int32_t *__restrict__ out_row, int32_t *__restrict__ out_col,
                                      float *__restrict__ out_val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t r = row[i];
    if (r < lo || r >= hi) return;
    const int64_t o = *cursor + (int64_t)pos[i];
    if (o >= capacity) return;
    out_row[o] = rebase ? (int32_t)(r - lo) : r;
    out_col[o] = col[i];
    if (out_val) out_val[o] = val ? val[i] : 1.0f;
}

__global__ void select_advance_kernel(int64_t *__restrict__ cursor, const uint32_t *__restrict__ total) {
    *cursor += (int64_t)*total;
}

// ------------------------------------------------------------------ chunks
__global__ void chunk_count_kernel(const int64_t *__restrict__ rowptr, int64_t n_rows, int32_t chunk_edges,
                                   int64_t *__restrict__ chunk_off, int64_t *__restrict__ heavy_off,
                                   int64_t *__restrict__ slot_off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t len = rowptr[i + 1] - rowptr[i];
    const int64_t nc = len <= chunk_edges ? 1 : (len + chunk_edges - 1) / chunk_edges;
    chunk_off[i] = nc;
    heavy_off[i] = nc > 1 ? 1 : 0;
    slot_off[i] = nc > 1 ? nc : 0;
}

__global__ void chunk_fill_kernel(const int64_t *__restrict__ rowptr, int64_t n_rows, int32_t chunk_edges,
                                  const int64_t *__restrict__ chunk_off, const int64_t *__restrict__ heavy_off,
                                  const int64_t *__restrict__ slot_off, int32_t *__restrict__ chunk_row,
                                  int64_t *__restrict__ chunk_begin, int32_t *__restrict__ chunk_slot,
                                  int32_t *__restrict__ heavy_row, int64_t *__restrict__ heavy_slot_ptr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t b = rowptr[i], len = rowptr[i + 1] - b;
    const int64_t nc = len <= chunk_edges ? 1 : (len + chunk_edges - 1) / chunk_edges;
    const int64_t c0 = chunk_off[i];
    const bool heavy = nc > 1;
    const int64_t s0 = slot_off[i];
    for (int64_t k = 0; k < nc; ++k) {
        chunk_row[c0 + k] = (int32_t)i;
        chunk_begin[c0 + k] = b + k * chunk_edges;
        chunk_slot[c0 + k] = heavy ? (int32_t)(s0 + k) : -1;
    }
    if (heavy) {
        const int64_t h = heavy_off[i];
        heavy_row[h] = (int32_t)i;
        heavy_slot_ptr[h] = s0;
        heavy_slot_ptr[h + 1] = s0 + nc;  // the next heavy row writes the same value
    }
}


// ------------------------------------------------------------------ column-blocked chunks
// Rows with at least block_min_len edges are cut where their (ascending) column ids cross a multiple of block_cols,
// and every such segment further into pieces of at most chunk_edges edges.  All their chunks are scheduled AFTER the
// ordinary rows' chunks and ordered by (column block, row): CTAs are dispatched in chunk order, so at any moment the
// resident warps gather from one window of block_cols operand rows, which stays in L2 (block_cols * D * 4 bytes)
// instead of streaming the whole operand table from HBM once per edge.  The cut points depend on the row's own
// column ids and on (block_cols, chunk_edges) only, so the reduction tree of a row - partials added in ascending
// column order by the heavy-row kernel - is the same on every launch shape and every row partition.
__device__ __forceinline__ int64_t lower_bound_col(const int32_t *__restrict__ colidx, int64_t lo, int64_t hi, int64_t key) {
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if ((int64_t)colidx[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void blocked_classify_kernel(const int64_t *__restrict__ rowptr, int64_t n_rows, int32_t chunk_edges,
                                        int32_t block_min_len, int64_t *__restrict__ chunk_off,
                                        int64_t *__restrict__ heavy_off, int64_t *__restrict__ slot_off,
                                        int64_t *__restrict__ blk_idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t len = rowptr[i + 1] - rowptr[i];
    const bool blocked = len >= block_min_len;
    const int64_t nc = len <= chunk_edges ? 1 : (len + chunk_edges - 1) / chunk_edges;
    blk_idx[i] = blocked ? 1 : 0;
    chunk_off[i] = blocked ? 0 : nc;
    heavy_off[i] = (blocked || nc > 1) ? 1 : 0;
    slot_off[i] = blocked ? 0 : (nc > 1 ? nc : 0);  // blocked rows: filled in by blocked_count_kernel
}

// hdr[0] = number of blocked rows (from the scan of the flags); mat is [n_blocks][hdr[0]], column-block major
__global__ void blocked_count_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ colidx, int64_t n_rows,
                                     int32_t chunk_edges, int32_t block_min_len, int64_t block_cols, int64_t n_blocks,
                                     const int64_t *__restrict__ blk_idx, const int64_t *__restrict__ hdr,
                                     int64_t *__restrict__ mat, int64_t *__restrict__ slot_off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t b = rowptr[i], e = rowptr[i + 1];
    if (e - b < block_min_len) return;
    const int64_t nb = hdr[0], j = blk_idx[i];
    int64_t lo = b, total = 0;
    for (int64_t cb = 0; cb < n_blocks; ++cb) {
        const int64_t hi = (cb + 1 == n_blocks) ? e : lower_bound_col(colidx, lo, e, (cb + 1) * block_cols);
        const int64_t n = (hi - lo + chunk_edges - 1) / chunk_edges;
        mat[cb * nb + j] = n;
        total += n;
        lo = hi;
    }
    slot_off[i] = total;
}

// ordinary rows exactly as chunk_fill_kernel (plus the explicit length); blocked rows only register as heavy
__global__ void blocked_fill_plain_kernel(const int64_t *__restrict__ rowptr, int64_t n_rows, int32_t chunk_edges,
                                          int32_t block_min_len, const int64_t *__restrict__ chunk_off,
                                          const int64_t *__restrict__ heavy_off, const int64_t *__restrict__ slot_off,
                                          int32_t *__restrict__ chunk_row,
                                          int64_t *__restrict__ chunk_begin, int32_t *__restrict__ chunk_len,
                                          int32_t *__restrict__ chunk_slot, int32_t *__restrict__ heavy_row,
                                          int64_t *__restrict__ heavy_slot_ptr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t b = rowptr[i], len = rowptr[i + 1] - b;
    const bool blocked = len >= block_min_len;
    const int64_t s0 = slot_off[i];
    if (!blocked) {
        const int64_t nc = len <= chunk_edges ? 1 : (len + chunk_edges - 1) / chunk_edges;
        const int64_t c0 = chunk_off[i];
        for (int64_t k = 0; k < nc; ++k) {
            const int64_t cb = b + k * chunk_edges;
            chunk_row[c0 + k] = (int32_t)i;
            chunk_begin[c0 + k] = cb;
            chunk_len[c0 + k] = (int32_t)((len - k * chunk_edges < chunk_edges) ? len - k * chunk_edges : chunk_edges);
            chunk_slot[c0 + k] = nc > 1 ? (int32_t)(s0 + k) : -1;
        }
        if (nc <= 1) return;
    }
    const int64_t h = heavy_off[i];
    heavy_row[h] = (int32_t)i;
    heavy_slot_ptr[h] = s0;
}

// heavy_slot_ptr[h + 1] for every heavy row = slot_off of the next heavy row, or the total for the last one: since
// slot_off is an exclusive scan over ALL rows and non-heavy rows contribute 0, slot_off[i + 1] is exactly that value
__global__ void blocked_fill_close_kernel(const int64_t *__restrict__ rowptr, int64_t n_rows, int32_t chunk_edges,
                                          int32_t block_min_len, const int64_t *__restrict__ heavy_off,
                                          const int64_t *__restrict__ slot_off, const int64_t *__restrict__ slot_total,
                                          int64_t *__restrict__ heavy_slot_ptr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t len = rowptr[i + 1] - rowptr[i];
    if (!(len >= block_min_len || len > chunk_edges)) return;
    heavy_slot_ptr[heavy_off[i] + 1] = (i + 1 < n_rows) ? slot_off[i + 1] : slot_total[0];
}

__global__ void blocked_fill_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ colidx, int64_t n_rows,
                                    int32_t chunk_edges, int32_t block_min_len, int64_t block_cols, int64_t n_blocks,
                                    const int64_t *__restrict__ blk_idx, const int64_t *__restrict__ hdr,
                                    const int64_t *__restrict__ mat, const int64_t *__restrict__ slot_off,
                                    int32_t *__restrict__ chunk_row, int64_t *__restrict__ chunk_begin,
                                    int32_t *__restrict__ chunk_len, int32_t *__restrict__ chunk_slot) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t b = rowptr[i], e = rowptr[i + 1];
    if (e - b < block_min_len) return;
    const int64_t nb = hdr[0], n_plain = hdr[1], j = blk_idx[i];
    int64_t lo = b, slot = slot_off[i];
    for (int64_t cb = 0; cb < n_blocks; ++cb) {
        const int64_t hi = (cb + 1 == n_blocks) ? e : lower_bound_col(colidx, lo, e, (cb + 1) * block_cols);
        int64_t pos = n_plain + mat[cb * nb + j];
        for (int64_t s = lo; s < hi; s += chunk_edges, ++pos, ++slot) {
            chunk_row[pos] = (int32_t)i;
            chunk_begin[pos] = s;
            chunk_len[pos] = (int32_t)((hi - s < chunk_edges) ? hi - s : chunk_edges);
            chunk_slot[pos] = (int32_t)slot;
        }
        lo = hi;
    }
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_graph_build_workspace_bytes(int64_t nnz, int64_t n_nodes, int flags) {
    return graph_ws_bytes(nnz, n_nodes, flags);
}

extern "C" int cbrs_graph_build_csr(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val, int64_t nnz,
                                    int64_t n_nodes, int flags, int64_t *rowptr, int32_t *colidx, float *vals,
                                    int64_t *nnz_out, void *workspace, size_t workspace_bytes, void *stream) {
    return build(coo_row, coo_col, nullptr, coo_val, nnz, 0, n_nodes, n_nodes, 1, 0, flags, rowptr, colidx, vals, nullptr,
                 nnz_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int cbrs_graph_build_csr_rel(const int32_t *coo_row, const int32_t *coo_col, const int32_t *coo_rel,
                                        const float *coo_val, int64_t nnz, int64_t n_nodes, int32_t n_rel,
                                        int32_t self_rel, int flags, int64_t *rowptr, int32_t *colidx, float *vals,
                                        int64_t *nnz_out, void *workspace, size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(coo_rel || n_rel == 1, CBRS_E_INVALID, "graph_build_rel: null relation ids");
    return build(coo_row, coo_col, coo_rel, coo_val, nnz, 0, n_nodes, n_nodes, n_rel, self_rel, flags, rowptr, colidx,
                 vals, nullptr, nnz_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- partitioned build (include/cbrs_b200.h) -------------------------------------------------------------------
extern "C" int cbrs_coo_row_histogram(const int32_t *coo_row, int64_t n, int64_t n_rows, int64_t *counts, void *stream) {
    CBRS_REQUIRE(n >= 0 && n_rows > 0 && counts && (coo_row || n == 0), CBRS_E_INVALID, "coo_row_histogram: bad argument");
    if (n == 0) return CBRS_OK;
    row_histogram_kernel<<<(unsigned)cdiv(n, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        coo_row, n, n_rows, (unsigned long long *)counts);
    CBRS_CHECK_LAUNCH("row_histogram");
    return CBRS_OK;
}

extern "C" size_t cbrs_coo_select_rows_workspace_bytes(int64_t n) {
    return align_up((size_t)(n > 0 ? n : 1) * 4) + 256 + scan_u32_workspace_bytes(n > 0 ? n : 1) + 1024;
}

extern "C" int cbrs_coo_select_rows(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val, int64_t n,
                                    int64_t row_lo, int64_t row_hi, int rebase, int32_t *out_row, int32_t *out_col,
                                    float *out_val, int64_t *cursor, int64_t capacity, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CBRS_REQUIRE(n >= 0 && (n == 0 || (coo_row && coo_col)) && out_row && out_col && cursor && capacity >= 0,
                 CBRS_E_INVALID, "coo_select_rows: bad argument");
    CBRS_REQUIRE(row_lo >= 0 && row_lo <= row_hi, CBRS_E_INVALID, "coo_select_rows: rows [%lld, %lld)", (long long)row_lo,
                 (long long)row_hi);
    CBRS_REQUIRE(n < (int64_t)0xfffffff0ll, CBRS_E_INVALID, "coo_select_rows: %lld entries exceed the 32-bit position range",
                 (long long)n);
    if (n == 0) return CBRS_OK;
    Arena a(workspace, workspace_bytes);
    uint32_t *pos = a.take<uint32_t>((size_t)n);
    uint32_t *total = a.take<uint32_t>(1);
    CBRS_REQUIRE(pos && total, CBRS_E_WORKSPACE, "coo_select_rows: workspace too small");
    void *sub = (char *)workspace + a.off;
    const size_t sub_bytes = workspace_bytes - a.off;
    const unsigned g = (unsigned)cdiv(n, kThreads);
    select_flags_kernel<<<g, kThreads, 0, s>>>(coo_row, n, row_lo, row_hi, pos);
    CBRS_CHECK_LAUNCH("select_flags");
    int rc = scan_u32_exclusive(pos, n, total, sub, sub_bytes, s);
    if (rc) return rc;
    select_scatter_kernel<<<g, kThreads, 0, s>>>(coo_row, coo_col, coo_val, n, row_lo, row_hi, rebase, pos, cursor, capacity,
                                                 out_row, out_col, out_val);
    CBRS_CHECK_LAUNCH("select_scatter");
    select_advance_kernel<<<1, 1, 0, s>>>(cursor, total);   // after the scatter: it reads the cursor
    CBRS_CHECK_LAUNCH("select_advance");
    return CBRS_OK;
}

extern "C" size_t cbrs_graph_build_block_workspace_bytes(int64_t nnz, int64_t n_rows, int flags) {
    return graph_ws_bytes(nnz, n_rows, flags);
}

extern "C" int cbrs_graph_build_block(const int32_t *coo_row, const int32_t *coo_col, const float *coo_val, int64_t nnz,
                                      int64_t row_lo, int64_t row_hi, int64_t n_cols, int flags, int64_t *rowptr,
                                      int32_t *colidx, float *vals, float *dinv_out, int64_t *nnz_out, void *workspace,
                                      size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(!(flags & CBRS_GRAPH_SYM_NORM) || dinv_out, CBRS_E_INVALID, "graph_build_block: SYM_NORM needs dinv_out");
    return build(coo_row, coo_col, nullptr, coo_val, nnz, row_lo, row_hi - row_lo, n_cols, 1, 0, flags, rowptr, colidx,
                 vals, (flags & CBRS_GRAPH_SYM_NORM) ? dinv_out : nullptr, nnz_out, workspace, workspace_bytes,
                 (cudaStream_t)stream);
}

extern "C" int cbrs_graph_block_scale(const int64_t *rowptr, const int32_t *colidx, float *vals, int64_t n_rows,
                                      int64_t row_lo, int64_t n_cols, const float *dinv, void *stream) {
    CBRS_REQUIRE(rowptr && colidx && vals && dinv && n_rows > 0 && row_lo >= 0 && row_lo + n_rows <= n_cols,
                 CBRS_E_INVALID, "graph_block_scale: bad argument");
    const unsigned gr = (unsigned)cdiv(n_rows * 32, kThreads);
    sym_scale_kernel<<<gr, kThreads, 0, (cudaStream_t)stream>>>(rowptr, colidx, dinv + row_lo, dinv, n_rows, n_cols, vals);
    CBRS_CHECK_LAUNCH("sym_scale");
    return CBRS_OK;
}

extern "C" size_t cbrs_chunks_workspace_bytes(int64_t n_rows) {
    return 3 * align_up((size_t)(n_rows > 0 ? n_rows : 1) * 8) + scan_i64_workspace_bytes(n_rows) + 1024;
}

static int chunk_arrays(void *ws, size_t ws_bytes, int64_t n_rows, int64_t **chunk_off, int64_t **heavy_off,
                        int64_t **slot_off, void **sub, size_t *sub_bytes) {
    Arena a(ws, ws_bytes);
    *chunk_off = a.take<int64_t>((size_t)n_rows);
    *heavy_off = a.take<int64_t>((size_t)n_rows);
    *slot_off = a.take<int64_t>((size_t)n_rows);
    CBRS_REQUIRE(*chunk_off && *heavy_off && *slot_off, CBRS_E_WORKSPACE, "chunks: workspace too small");
    *sub = (char *)ws + a.off;
    *sub_bytes = ws_bytes - a.off;
    return CBRS_OK;
}

extern "C" int cbrs_chunks_count(const int64_t *rowptr, int64_t n_rows, int32_t chunk_edges, int64_t *counts_out,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CBRS_REQUIRE(rowptr && counts_out && n_rows > 0 && chunk_edges > 0, CBRS_E_INVALID, "chunks_count: bad argument");
    int64_t *chunk_off, *heavy_off, *slot_off;
    void *sub;
    size_t sub_bytes;
    int rc = chunk_arrays(workspace, workspace_bytes, n_rows, &chunk_off, &heavy_off, &slot_off, &sub, &sub_bytes);
    if (rc) return rc;
    chunk_count_kernel<<<(unsigned)cdiv(n_rows, kThreads), kThreads, 0, s>>>(rowptr, n_rows, chunk_edges, chunk_off,
                                                                            heavy_off, slot_off);
    CBRS_CHECK_LAUNCH("chunk_count");
    if ((rc = scan_i64_exclusive(chunk_off, n_rows, counts_out + 0, sub, sub_bytes, s))) return rc;
    if ((rc = scan_i64_exclusive(heavy_off, n_rows, counts_out + 1, sub, sub_bytes, s))) return rc;
    if ((rc = scan_i64_exclusive(slot_off, n_rows, counts_out + 2, sub, sub_bytes, s))) return rc;
    return CBRS_OK;
}

extern "C" int cbrs_chunks_fill(const int64_t *rowptr, int64_t n_rows, int32_t chunk_edges, int32_t *chunk_row,
                                int64_t *chunk_begin, int32_t *chunk_slot, int32_t *heavy_row,
                                int64_t *heavy_slot_ptr, void *workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CBRS_REQUIRE(rowptr && chunk_row && chunk_begin && chunk_slot && n_rows > 0 && chunk_edges > 0, CBRS_E_INVALID,
                 "chunks_fill: bad argument");
    int64_t *chunk_off, *heavy_off, *slot_off;
    void *sub;
    size_t sub_bytes;
    int rc = chunk_arrays(workspace, workspace_bytes, n_rows, &chunk_off, &heavy_off, &slot_off, &sub, &sub_bytes);
    if (rc) return rc;
    chunk_fill_kernel<<<(unsigned)cdiv(n_rows, kThreads), kThreads, 0, s>>>(
        rowptr, n_rows, chunk_edges, chunk_off, heavy_off, slot_off, chunk_row, chunk_begin, chunk_slot, heavy_row,
        heavy_slot_ptr);
    CBRS_CHECK_LAUNCH("chunk_fill");
    return CBRS_OK;
}

// ---- column-blocked decomposition (see the kernels above) -------------------------------------------------
static int64_t blocked_rows_bound(int64_t n_rows, int64_t nnz, int32_t block_min_len) {
    const int64_t by_len = nnz / (block_min_len > 0 ? block_min_len : 1);
    return by_len < n_rows ? by_len : n_rows;
}

extern "C" size_t cbrs_chunks_blocked_workspace_bytes(int64_t n_rows, int64_t nnz, int64_t n_cols, int32_t block_min_len,
                                                      int64_t block_cols) {
    if (n_rows <= 0) n_rows = 1;
    const int64_t n_blocks = block_cols > 0 ? cdiv(n_cols > 0 ? n_cols : 1, block_cols) : 1;
    const int64_t mat = blocked_rows_bound(n_rows, nnz, block_min_len) * n_blocks + 1;
    return 4 * align_up((size_t)n_rows * 8) + align_up((size_t)mat * 8) + align_up(64) +
           scan_i64_workspace_bytes(mat > n_rows ? mat : n_rows) + 1024;
}

namespace {
struct BlockedWs {
    int64_t *chunk_off, *heavy_off, *slot_off, *blk_idx, *mat, *hdr;  // hdr: {n_blocked, n_plain_chunks, n_slots, n_mat}
    void *sub;
    size_t sub_bytes;
    int64_t mat_cap;
};
}  // namespace

static int blocked_arrays(void *ws, size_t ws_bytes, int64_t n_rows, int64_t nnz, int64_t n_cols, int32_t block_min_len,
                          int64_t block_cols, BlockedWs *w) {
    Arena a(ws, ws_bytes);
    const int64_t n_blocks = cdiv(n_cols, block_cols);
    w->mat_cap = blocked_rows_bound(n_rows, nnz, block_min_len) * n_blocks + 1;
    w->chunk_off = a.take<int64_t>((size_t)n_rows);
    w->heavy_off = a.take<int64_t>((size_t)n_rows);
    w->slot_off = a.take<int64_t>((size_t)n_rows);
    w->blk_idx = a.take<int64_t>((size_t)n_rows);
    w->mat = a.take<int64_t>((size_t)w->mat_cap);
    w->hdr = a.take<int64_t>(8);
    CBRS_REQUIRE(w->chunk_off && w->heavy_off && w->slot_off && w->blk_idx && w->mat && w->hdr, CBRS_E_WORKSPACE,
                 "chunks_blocked: workspace too small");
    w->sub = (char *)ws + a.off;
    w->sub_bytes = ws_bytes - a.off;
    return CBRS_OK;
}

extern "C" int cbrs_chunks_blocked_count(const int64_t *rowptr, const int32_t *colidx, int64_t n_rows, int64_t nnz,
                                         int64_t n_cols, int32_t chunk_edges, int32_t block_min_len, int64_t block_cols,
                                         int64_t *counts_out, void *workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CBRS_REQUIRE(rowptr && counts_out && n_rows > 0 && chunk_edges > 0 && (colidx || nnz == 0), CBRS_E_INVALID,
                 "chunks_blocked_count: bad argument");
    CBRS_REQUIRE(block_cols > 0 && block_min_len > 0 && n_cols > 0, CBRS_E_INVALID,
                 "chunks_blocked_count: block_cols=%lld block_min_len=%d n_cols=%lld", (long long)block_cols, block_min_len,
                 (long long)n_cols);
    BlockedWs w;
    int rc = blocked_arrays(workspace, workspace_bytes, n_rows, nnz, n_cols, block_min_len, block_cols, &w);
    if (rc) return rc;
    const int64_t n_blocks = cdiv(n_cols, block_cols);
    const unsigned grid = (unsigned)cdiv(n_rows, kThreads);
    blocked_classify_kernel<<<grid, kThreads, 0, s>>>(rowptr, n_rows, chunk_edges, block_min_len, w.chunk_off, w.heavy_off,
                                                      w.slot_off, w.blk_idx);
    CBRS_CHECK_LAUNCH("blocked_classify");
    if ((rc = scan_i64_exclusive(w.blk_idx, n_rows, w.hdr + 0, w.sub, w.sub_bytes, s))) return rc;
    // the matrix is sized by the number of blocked rows: one host round trip (graph build is not a hot path)
    int64_t n_blocked = 0;
    cudaError_t e = cudaMemcpyAsync(&n_blocked, w.hdr + 0, 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "chunks_blocked_count: %s", cudaGetErrorString(e));
    const int64_t n_mat = n_blocked * n_blocks;
    CBRS_REQUIRE(n_mat < w.mat_cap, CBRS_E_WORKSPACE, "chunks_blocked_count: %lld blocked rows exceed the bound",
                 (long long)n_blocked);
    if (n_blocked > 0) {
        blocked_count_kernel<<<grid, kThreads, 0, s>>>(rowptr, colidx, n_rows, chunk_edges, block_min_len, block_cols,
                                                       n_blocks, w.blk_idx, w.hdr, w.mat, w.slot_off);
        CBRS_CHECK_LAUNCH("blocked_count");
    }
    if ((rc = scan_i64_exclusive(w.chunk_off, n_rows, w.hdr + 1, w.sub, w.sub_bytes, s))) return rc;
    if ((rc = scan_i64_exclusive(w.heavy_off, n_rows, counts_out + 1, w.sub, w.sub_bytes, s))) return rc;
    if ((rc = scan_i64_exclusive(w.slot_off, n_rows, w.hdr + 2, w.sub, w.sub_bytes, s))) return rc;
    e = cudaMemsetAsync(w.hdr + 3, 0, 8, s);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "chunks_blocked_count: %s", cudaGetErrorString(e));
    if (n_mat > 0 && (rc = scan_i64_exclusive(w.mat, n_mat, w.hdr + 3, w.sub, w.sub_bytes, s))) return rc;
    // counts_out = {plain + blocked chunks, heavy rows, slots}
    int64_t h[4];
    e = cudaMemcpyAsync(h, w.hdr, 32, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "chunks_blocked_count: %s", cudaGetErrorString(e));
    const int64_t total = h[1] + h[3];
    e = cudaMemcpyAsync(counts_out + 0, &total, 8, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(counts_out + 2, w.hdr + 2, 8, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // `total` lives on this stack frame
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "chunks_blocked_count: %s", cudaGetErrorString(e));
    return CBRS_OK;
}

extern "C" int cbrs_chunks_blocked_fill(const int64_t *rowptr, const int32_t *colidx, int64_t n_rows, int64_t nnz,
                                        int64_t n_cols, int32_t chunk_edges, int32_t block_min_len, int64_t block_cols,
                                        int32_t *chunk_row, int64_t *chunk_begin, int32_t *chunk_len, int32_t *chunk_slot,
                                        int32_t *heavy_row, int64_t *heavy_slot_ptr, void *workspace,
                                        size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CBRS_REQUIRE(rowptr && chunk_row && chunk_begin && chunk_len && chunk_slot && n_rows > 0 && chunk_edges > 0 &&
                     (colidx || nnz == 0),
                 CBRS_E_INVALID, "chunks_blocked_fill: bad argument");
    CBRS_REQUIRE(block_cols > 0 && block_min_len > 0 && n_cols > 0, CBRS_E_INVALID, "chunks_blocked_fill: bad blocking");
    BlockedWs w;
    int rc = blocked_arrays(workspace, workspace_bytes, n_rows, nnz, n_cols, block_min_len, block_cols, &w);
    if (rc) return rc;
    const int64_t n_blocks = cdiv(n_cols, block_cols);
    const unsigned grid = (unsigned)cdiv(n_rows, kThreads);
    blocked_fill_plain_kernel<<<grid, kThreads, 0, s>>>(rowptr, n_rows, chunk_edges, block_min_len, w.chunk_off, w.heavy_off,
                                                        w.slot_off, chunk_row, chunk_begin, chunk_len, chunk_slot, heavy_row,
                                                        heavy_slot_ptr);
    CBRS_CHECK_LAUNCH("blocked_fill_plain");
    if (heavy_slot_ptr) {
        blocked_fill_close_kernel<<<grid, kThreads, 0, s>>>(rowptr, n_rows, chunk_edges, block_min_len, w.heavy_off,
                                                            w.slot_off, w.hdr + 2, heavy_slot_ptr);
        CBRS_CHECK_LAUNCH("blocked_fill_close");
    }
    blocked_fill_kernel<<<grid, kThreads, 0, s>>>(rowptr, colidx, n_rows, chunk_edges, block_min_len, block_cols, n_blocks,
                                                  w.blk_idx, w.hdr, w.mat, w.slot_off, chunk_row, chunk_begin, chunk_len,
                                                  chunk_slot);
    CBRS_CHECK_LAUNCH("blocked_fill");
    return CBRS_OK;
}
