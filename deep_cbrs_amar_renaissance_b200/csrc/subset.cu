// Row-subset work decomposition: the chunks of a set of needed rows, taken from a full cbrs_csr_t.
//
// The per-batch model call reads its last layer's output only at the batch's rows.  The subset keeps the full
// descriptor's rowptr/colidx/vals and chunk geometry and lists only the needed rows' chunks, in their original list
// order (so the column-blocked (window, row) order of heavy rows is kept); the needed heavy rows keep their slot
// order, renumbered compactly.  The propagation kernels then compute every needed row with the same chunks, in the
// same order, with the same partial merge tree as the full launch: the same bits.
#include "common.cuh"

namespace cbrs {

namespace {
constexpr int kSubThreads = 256;

struct SubsetWs {
    uint32_t *row_flag;   // [n_rows]   1 = needed
    uint32_t *chunk_pos;  // [n_chunks] flag, then its exclusive scan = position in the subset
    uint32_t *slot_pos;   // [n_slots]  flag, then its exclusive scan = renumbered slot
    uint32_t *heavy_pos;  // [n_heavy]  flag, then its exclusive scan = position in the subset's heavy list
    uint32_t *tot;        // {chunks, slots, heavy rows}
    unsigned long long *work;  // {distinct needed rows, their edges}
    void *sub;
    size_t sub_bytes;
};

int64_t max4(int64_t a, int64_t b, int64_t c, int64_t d) {
    const int64_t x = a > b ? a : b, y = c > d ? c : d;
    return x > y ? x : y;
}
}  // namespace

__global__ void subset_mark_rows_kernel(const int64_t *__restrict__ ids, int64_t n_ids, int64_t n_rows,
                                        const int64_t *__restrict__ rowptr, uint32_t *__restrict__ row_flag,
                                        unsigned long long *__restrict__ work) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_ids) return;
    const int64_t r = ids[k];
    if (r < 0 || r >= n_rows) return;  // ids outside the table select nothing
    if (atomicExch(row_flag + r, 1u) == 0u) {  // first id of this row: count it once
        atomicAdd(work + 0, 1ull);
        atomicAdd(work + 1, (unsigned long long)(rowptr[r + 1] - rowptr[r]));
    }
}

__global__ void subset_flag_chunks_kernel(const int32_t *__restrict__ chunk_row, const int32_t *__restrict__ chunk_slot,
                                          int64_t n_chunks, const uint32_t *__restrict__ row_flag,
                                          uint32_t *__restrict__ chunk_pos, uint32_t *__restrict__ slot_pos) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const uint32_t f = row_flag[chunk_row[c]];
    chunk_pos[c] = f;
    const int32_t s = chunk_slot[c];
    if (s >= 0) slot_pos[s] = f;  // every slot belongs to exactly one chunk
}

__global__ void subset_flag_heavy_kernel(const int32_t *__restrict__ heavy_row, int64_t n_heavy,
                                         const uint32_t *__restrict__ row_flag, uint32_t *__restrict__ heavy_pos) {
    const int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h < n_heavy) heavy_pos[h] = row_flag[heavy_row[h]];
}

__global__ void subset_counts_kernel(const uint32_t *__restrict__ tot, const unsigned long long *__restrict__ work,
                                     int64_t *__restrict__ counts_out) {
    counts_out[0] = tot[0];
    counts_out[1] = tot[2];
    counts_out[2] = tot[1];
    counts_out[3] = (int64_t)work[0];
    counts_out[4] = (int64_t)work[1];
}

__global__ void subset_fill_chunks_kernel(const int32_t *__restrict__ chunk_row, const int64_t *__restrict__ chunk_begin,
                                          const int32_t *__restrict__ chunk_len, const int32_t *__restrict__ chunk_slot,
                                          int64_t n_chunks, const uint32_t *__restrict__ row_flag,
                                          const uint32_t *__restrict__ chunk_pos, const uint32_t *__restrict__ slot_pos,
                                          int32_t *__restrict__ o_row, int64_t *__restrict__ o_begin,
                                          int32_t *__restrict__ o_len, int32_t *__restrict__ o_slot) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const int32_t row = chunk_row[c];
    if (!row_flag[row]) return;
    const uint32_t o = chunk_pos[c];
    const int32_t s = chunk_slot[c];
    o_row[o] = row;
    o_begin[o] = chunk_begin[c];
    if (chunk_len) o_len[o] = chunk_len[c];
    o_slot[o] = s >= 0 ? (int32_t)slot_pos[s] : -1;
}

// a needed heavy row's slots [s0, s1) are all needed, so they stay contiguous and in order: [slot_pos[s0], + s1 - s0)
__global__ void subset_fill_heavy_kernel(const int32_t *__restrict__ heavy_row, const int64_t *__restrict__ heavy_slot_ptr,
                                         int64_t n_heavy, const uint32_t *__restrict__ row_flag,
                                         const uint32_t *__restrict__ heavy_pos, const uint32_t *__restrict__ slot_pos,
                                         const uint32_t *__restrict__ tot, int32_t *__restrict__ o_heavy_row,
                                         int64_t *__restrict__ o_heavy_slot_ptr) {
    const int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n_heavy) return;
    const int32_t row = heavy_row[h];
    if (!row_flag[row]) return;
    const uint32_t o = heavy_pos[h];
    const int64_t s0 = heavy_slot_ptr[h], s1 = heavy_slot_ptr[h + 1];
    const int64_t n0 = s1 > s0 ? (int64_t)slot_pos[s0] : (int64_t)tot[1];
    o_heavy_row[o] = row;
    o_heavy_slot_ptr[o] = n0;
    o_heavy_slot_ptr[o + 1] = n0 + (s1 - s0);  // the next needed heavy row writes the same value
}

static int subset_arrays(const cbrs_csr_t *g, void *ws, size_t ws_bytes, SubsetWs *w) {
    Arena a(ws, ws_bytes);
    w->row_flag = a.take<uint32_t>((size_t)(g->n_rows > 0 ? g->n_rows : 1));
    w->chunk_pos = a.take<uint32_t>((size_t)(g->n_chunks > 0 ? g->n_chunks : 1));
    w->slot_pos = a.take<uint32_t>((size_t)(g->n_slots > 0 ? g->n_slots : 1));
    w->heavy_pos = a.take<uint32_t>((size_t)(g->n_heavy > 0 ? g->n_heavy : 1));
    w->tot = a.take<uint32_t>(4);
    w->work = a.take<unsigned long long>(2);
    CBRS_REQUIRE(w->row_flag && w->chunk_pos && w->slot_pos && w->heavy_pos && w->tot && w->work, CBRS_E_WORKSPACE,
                 "csr_subset: workspace too small");
    w->sub = (char *)ws + a.off;
    w->sub_bytes = ws_bytes - a.off;
    return CBRS_OK;
}

static int check_desc(const cbrs_csr_t *g, const char *what) {
    CBRS_REQUIRE(g && g->n_rows > 0 && g->n_chunks >= 0 && g->n_heavy >= 0 && g->n_slots >= 0, CBRS_E_INVALID,
                 "%s: bad graph descriptor", what);
    CBRS_REQUIRE(g->n_chunks < (int64_t)0xffffffffll && g->n_slots < (int64_t)0xffffffffll, CBRS_E_INVALID,
                 "%s: %lld chunks / %lld slots exceed the 32-bit position range", what, (long long)g->n_chunks,
                 (long long)g->n_slots);
    CBRS_REQUIRE(g->rowptr && g->chunk_row && g->chunk_begin && g->chunk_slot && (g->n_heavy == 0 || (g->heavy_row && g->heavy_slot_ptr)),
                 CBRS_E_INVALID, "%s: graph descriptor has null arrays", what);
    return CBRS_OK;
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_csr_subset_workspace_bytes(const cbrs_csr_t *g) {
    if (!g) return 0;
    const int64_t n = max4(g->n_rows, g->n_chunks, g->n_slots, g->n_heavy);
    return align_up((size_t)(g->n_rows > 0 ? g->n_rows : 1) * 4) + align_up((size_t)(g->n_chunks > 0 ? g->n_chunks : 1) * 4) +
           align_up((size_t)(g->n_slots > 0 ? g->n_slots : 1) * 4) + align_up((size_t)(g->n_heavy > 0 ? g->n_heavy : 1) * 4) +
           align_up(16) + align_up(16) + scan_u32_workspace_bytes(n > 0 ? n : 1) + 1024;
}

extern "C" int cbrs_csr_subset_count(const cbrs_csr_t *g, const int64_t *ids, int64_t n_ids, int64_t *counts_out,
                                     void *workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    int rc = check_desc(g, "csr_subset_count");
    if (rc) return rc;
    CBRS_REQUIRE(counts_out && n_ids >= 0 && (ids || n_ids == 0), CBRS_E_INVALID, "csr_subset_count: bad argument");
    SubsetWs w;
    if ((rc = subset_arrays(g, workspace, workspace_bytes, &w))) return rc;
    cudaError_t e = cudaMemsetAsync(w.row_flag, 0, (size_t)g->n_rows * 4, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(w.tot, 0, 16, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(w.work, 0, 16, s);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "csr_subset_count: %s", cudaGetErrorString(e));
    if (n_ids > 0) {
        subset_mark_rows_kernel<<<(unsigned)cdiv(n_ids, kSubThreads), kSubThreads, 0, s>>>(ids, n_ids, g->n_rows, g->rowptr,
                                                                                          w.row_flag, w.work);
        CBRS_CHECK_LAUNCH("subset_mark_rows");
    }
    if (g->n_chunks > 0) {
        subset_flag_chunks_kernel<<<(unsigned)cdiv(g->n_chunks, kSubThreads), kSubThreads, 0, s>>>(
            g->chunk_row, g->chunk_slot, g->n_chunks, w.row_flag, w.chunk_pos, w.slot_pos);
        CBRS_CHECK_LAUNCH("subset_flag_chunks");
        if ((rc = scan_u32_exclusive(w.chunk_pos, g->n_chunks, w.tot + 0, w.sub, w.sub_bytes, s))) return rc;
    }
    if (g->n_slots > 0 && (rc = scan_u32_exclusive(w.slot_pos, g->n_slots, w.tot + 1, w.sub, w.sub_bytes, s))) return rc;
    if (g->n_heavy > 0) {
        subset_flag_heavy_kernel<<<(unsigned)cdiv(g->n_heavy, kSubThreads), kSubThreads, 0, s>>>(g->heavy_row, g->n_heavy,
                                                                                                w.row_flag, w.heavy_pos);
        CBRS_CHECK_LAUNCH("subset_flag_heavy");
        if ((rc = scan_u32_exclusive(w.heavy_pos, g->n_heavy, w.tot + 2, w.sub, w.sub_bytes, s))) return rc;
    }
    subset_counts_kernel<<<1, 1, 0, s>>>(w.tot, w.work, counts_out);
    CBRS_CHECK_LAUNCH("subset_counts");
    return CBRS_OK;
}

extern "C" int cbrs_csr_subset_fill(const cbrs_csr_t *g, int32_t *chunk_row, int64_t *chunk_begin, int32_t *chunk_len,
                                    int32_t *chunk_slot, int32_t *heavy_row, int64_t *heavy_slot_ptr, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    int rc = check_desc(g, "csr_subset_fill");
    if (rc) return rc;
    CBRS_REQUIRE(chunk_row && chunk_begin && chunk_slot && heavy_slot_ptr && (chunk_len || !g->chunk_len) &&
                     (heavy_row || g->n_heavy == 0),
                 CBRS_E_INVALID, "csr_subset_fill: null output");
    SubsetWs w;
    if ((rc = subset_arrays(g, workspace, workspace_bytes, &w))) return rc;
    if (g->n_chunks > 0) {
        subset_fill_chunks_kernel<<<(unsigned)cdiv(g->n_chunks, kSubThreads), kSubThreads, 0, s>>>(
            g->chunk_row, g->chunk_begin, g->chunk_len, g->chunk_slot, g->n_chunks, w.row_flag, w.chunk_pos, w.slot_pos,
            chunk_row, chunk_begin, chunk_len, chunk_slot);
        CBRS_CHECK_LAUNCH("subset_fill_chunks");
    }
    if (g->n_heavy > 0) {
        subset_fill_heavy_kernel<<<(unsigned)cdiv(g->n_heavy, kSubThreads), kSubThreads, 0, s>>>(
            g->heavy_row, g->heavy_slot_ptr, g->n_heavy, w.row_flag, w.heavy_pos, w.slot_pos, w.tot, heavy_row,
            heavy_slot_ptr);
        CBRS_CHECK_LAUNCH("subset_fill_heavy");
    }
    return CBRS_OK;
}
