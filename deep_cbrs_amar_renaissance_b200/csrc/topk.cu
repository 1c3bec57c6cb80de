// Per-user top-k.  Row T of SURVEY.md section 8a.
//
// Catalog form: the reference never scores the full catalog (it ranks only the test
// pairs, /root/reference/src/experiment.py:197-207); parity is defined as "reference
// scorer on every (u,i) + stable descending sort", i.e. ties go to the LOWER item index.
// Pair-list form: restates src/utilities/metrics.py:21-34 (pandas stable sort by
// (user asc, score desc), head(k) per user) with the stable device radix sort.
#include "common.cuh"

namespace cbrs {

constexpr int kTopkThreads = 256;

// One CTA per user.  Candidates are 64-bit keys (score bits high, ~item low) so "better"
// is a single unsigned compare and the lower item wins a score tie.  Round r extracts the
// largest key strictly below round r-1's winner; the score row stays in L1/L2.
__global__ void __launch_bounds__(kTopkThreads) topk_rows_kernel(const float *__restrict__ scores, int64_t ld,
                                                               int32_t n_items, int32_t k, int32_t *__restrict__ ids_out,
                                                               float *__restrict__ vals_out) {
    __shared__ unsigned long long warp_best[kTopkThreads / 32];
    __shared__ unsigned long long winner;
    const float *row = scores + (int64_t)blockIdx.x * ld;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long bound = ~0ull;  // exclusive upper bound
    for (int r = 0; r < k; ++r) {
        unsigned long long best = 0ull;  // 0 is below every real key
        for (int i = threadIdx.x; i < n_items; i += kTopkThreads) {
            const unsigned long long key = topk_key(row[i], (uint32_t)i);
            if (key < bound && key > best) best = key;
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o);
            best = t > best ? t : best;
        }
        if (lane == 0) warp_best[warp] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = warp_best[0];
#pragma unroll
            for (int w = 1; w < kTopkThreads / 32; ++w) b = warp_best[w] > b ? warp_best[w] : b;
            winner = b;
            const int64_t o = (int64_t)blockIdx.x * k + r;
            topk_store<false>(b, ids_out + o, vals_out + o);   // b = 0: fewer than k items
        }
        __syncthreads();
        bound = winner;
        if (bound == 0ull) bound = 0ull;  // nothing left: later rounds also emit -1
    }
}

__global__ void pair_keys_kernel(const int64_t *__restrict__ users, const float *__restrict__ scores, int64_t n,
                                 uint64_t *__restrict__ keys, uint32_t *__restrict__ payload) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // ascending key == (user asc, score desc); the stable sort keeps input order on ties
    keys[i] = ((uint64_t)users[i] << 32) | (uint64_t)(~orderable_f32(scores[i]));
    payload[i] = (uint32_t)i;
}

__global__ void pair_rank_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ payload, int64_t n,
                                 int32_t *__restrict__ order_out, int32_t *__restrict__ rank_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    order_out[i] = (int32_t)payload[i];
    const uint64_t u = keys[i] >> 32;
    if (i == 0 || (keys[i - 1] >> 32) != u) {  // run head numbers its run
        int32_t r = 0;
        for (int64_t j = i; j < n && (keys[j] >> 32) == u; ++j) rank_out[j] = r++;
    }
}

// Generic catalog path: one warp per row writes -inf over the listed items that fall in the row's column block
// [col_base, col_base + n_cols).  A binary search finds the first entry >= col_base; the lanes then walk the entries
// inside the block only, so a row costs log2(len) + (its items in the block) / 32 reads.
constexpr int kExclThreads = 256;
__global__ void __launch_bounds__(kExclThreads) exclude_cols_kernel(float *__restrict__ scores, int64_t ld, int64_t n_rows,
                                                                   int32_t n_cols, int32_t col_base,
                                                                   const int64_t *__restrict__ rowptr,
                                                                   const int32_t *__restrict__ items) {
    const int64_t r = (int64_t)blockIdx.x * (kExclThreads / 32) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int64_t end = __ldg(rowptr + r + 1);
    int64_t lo = __ldg(rowptr + r), hi = end;
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(items + mid) < col_base) lo = mid + 1; else hi = mid;
    }
    for (int64_t j = lo + lane; j < end; j += 32) {
        const int64_t c = (int64_t)__ldg(items + j) - col_base;
        if (c >= n_cols) break;   // sorted row: every later entry of this lane is past the block too
        if (c >= 0) scores[r * ld + c] = -INFINITY;
    }
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_exclude_cols(float *scores, int64_t ld, int64_t n_rows, int32_t n_cols, int32_t col_base,
                                 const int64_t *excl_rowptr, const int32_t *excl_items, void *stream) {
    CBRS_REQUIRE(scores, CBRS_E_INVALID, "exclude_cols: null scores");
    CBRS_REQUIRE(!excl_rowptr == !excl_items, CBRS_E_INVALID, "exclude_cols: %s is null but %s is not",
                 excl_rowptr ? "excl_items" : "excl_rowptr", excl_rowptr ? "excl_rowptr" : "excl_items");
    CBRS_REQUIRE(n_rows >= 0 && n_cols >= 0 && ld >= n_cols && col_base >= 0, CBRS_E_INVALID,
                 "exclude_cols: n_rows=%lld n_cols=%d ld=%lld col_base=%d", (long long)n_rows, n_cols, (long long)ld, col_base);
    if (!excl_rowptr || n_rows == 0 || n_cols == 0) return CBRS_OK;
    exclude_cols_kernel<<<(unsigned)cdiv(n_rows, kExclThreads / 32), kExclThreads, 0, (cudaStream_t)stream>>>(
        scores, ld, n_rows, n_cols, col_base, excl_rowptr, excl_items);
    CBRS_CHECK_LAUNCH("exclude_cols");
    return CBRS_OK;
}

extern "C" int cbrs_topk_rows(const float *scores, int64_t ld, int64_t n_users, int32_t n_items, int32_t k,
                              int32_t *ids_out, float *vals_out, void *stream) {
    CBRS_REQUIRE(scores && ids_out && vals_out, CBRS_E_INVALID, "topk_rows: null argument");
    CBRS_REQUIRE(n_users >= 0 && n_items > 0 && ld >= n_items && k > 0 && k <= 128, CBRS_E_INVALID,
                 "topk_rows: n_users=%lld n_items=%d k=%d", (long long)n_users, n_items, k);
    if (n_users == 0) return CBRS_OK;
    topk_rows_kernel<<<(unsigned)n_users, kTopkThreads, 0, (cudaStream_t)stream>>>(scores, ld, n_items, k, ids_out, vals_out);
    CBRS_CHECK_LAUNCH("topk_rows");
    return CBRS_OK;
}

extern "C" size_t cbrs_topk_pairs_workspace_bytes(int64_t n_pairs) {
    return align_up((size_t)n_pairs * 8) + align_up((size_t)n_pairs * 4) + sort_workspace_bytes(n_pairs) + 1024;
}

extern "C" int cbrs_topk_pairs(const int64_t *users, const float *scores, int64_t n_pairs, int64_t n_users,
                               int32_t *order_out, int32_t *rank_out, void *workspace, size_t workspace_bytes,
                               void *stream) {
    CBRS_REQUIRE(users && scores && order_out && rank_out, CBRS_E_INVALID, "topk_pairs: null argument");
    CBRS_REQUIRE(n_pairs >= 0 && n_pairs < ((int64_t)1 << 31) && n_users > 0 && n_users < ((int64_t)1 << 31),
                 CBRS_E_INVALID, "topk_pairs: n_pairs=%lld n_users=%lld", (long long)n_pairs, (long long)n_users);
    if (n_pairs == 0) return CBRS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    Arena a(workspace, workspace_bytes);
    uint64_t *keys = a.take<uint64_t>((size_t)n_pairs);
    uint32_t *payload = a.take<uint32_t>((size_t)n_pairs);
    CBRS_REQUIRE(keys && payload, CBRS_E_WORKSPACE, "topk_pairs: workspace too small");
    const unsigned g = (unsigned)cdiv(n_pairs, 256);
    pair_keys_kernel<<<g, 256, 0, s>>>(users, scores, n_pairs, keys, payload);
    CBRS_CHECK_LAUNCH("pair_keys");
    int user_bits = 1;
    while (((int64_t)1 << user_bits) < n_users) ++user_bits;
    int rc = sort_pairs_u64(keys, payload, n_pairs, 32 + user_bits, (char *)workspace + a.off, workspace_bytes - a.off, s);
    if (rc) return rc;
    pair_rank_kernel<<<g, 256, 0, s>>>(keys, payload, n_pairs, order_out, rank_out);
    CBRS_CHECK_LAUNCH("pair_rank");
    return CBRS_OK;
}
