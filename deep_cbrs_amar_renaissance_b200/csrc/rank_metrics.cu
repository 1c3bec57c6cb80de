// Full-catalog ranking metrics (P, R, HR, MRR, NDCG, AP at up to 8 cutoffs) of top-k lists against per-user relevance
// lists, all on the device: only n_cutoffs x 7 fp64 sums leave it.  Contract and definitions: include/cbrs_b200.h, above
// cbrs_rank_metrics.
//
// One warp per list.  Lane l holds slots l, l + 32, l + 64, l + 96 (k <= 128) and looks each id up in the user's
// relevance row with excluded_item's bounded binary search; four ballots then give every lane the whole hit mask, so
// hit counts and the first hit are popc / ffs of masked ballots.  The position-weighted sums (DCG, IDCG, AP) are lane
// partials reduced by an xor butterfly: every lane adds the same two values in commutative order, so all lanes hold the
// same bits, and the order depends on nothing but the slot positions.
//
// Determinism: block b always covers rows [b * kRmRowsPerBlock, (b + 1) * kRmRowsPerBlock), each warp adds its rows in row
// order, the warps are added in warp order, and the second launch adds the block partials of each value in a fixed
// strided-then-tree order.  The sums depend on n_rows and the data only: bit-identical from run to run, for any ld.
#include "common.cuh"

namespace cbrs {

constexpr int kRmWarps = 8;
constexpr int kRmRowsPerWarp = 16;
constexpr int kRmRowsPerBlock = kRmWarps * kRmRowsPerWarp;
constexpr int kRmMaxCutoffs = 8;
constexpr int kRmCols = 7;          // P, R, HR, MRR, NDCG, AP, users counted
constexpr int kRmPerUser = 6;
constexpr int kRmReduceThreads = 256;

struct Cutoffs {
    int32_t c[kRmMaxCutoffs];
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// partials: [n_cutoffs * 7][n_blocks]
__global__ void __launch_bounds__(kRmWarps * 32) rank_metrics_kernel(
    const int32_t *__restrict__ ids, int64_t ld, int64_t n_rows, int32_t k, int32_t n_items,
    const int64_t *__restrict__ users, int64_t n_users, const int64_t *__restrict__ rel_rowptr,
    const int32_t *__restrict__ rel_items, Cutoffs cut, int32_t n_cutoffs, double *__restrict__ per_user,
    double *__restrict__ partials) {
    __shared__ double warp_acc[kRmWarps][kRmMaxCutoffs * kRmCols];
    __shared__ int32_t cutoff[kRmMaxCutoffs];   // indexed by a loop counter: from shared memory, not a local copy
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < kRmMaxCutoffs; ++i) cutoff[i] = cut.c[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_vals = n_cutoffs * kRmCols;
    // lane l accumulates values l and l + 32 of the [n_cutoffs][7] table
    double acc0 = 0.0, acc1 = 0.0;
    // slot weights 1 / log2(r + 2) of this lane's four slots
    double w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = 1.0 / log2((double)(32 * j + lane + 2));

    const int64_t row0 = (int64_t)blockIdx.x * kRmRowsPerBlock + (int64_t)warp * kRmRowsPerWarp;
    for (int i = 0; i < kRmRowsPerWarp; ++i) {
        const int64_t row = row0 + i;
        if (row >= n_rows) break;
        const int64_t u = users ? __ldg(users + row) : row;
        int64_t n_rel = 0;
        if (rel_rowptr != nullptr && u >= 0 && u < n_users) n_rel = __ldg(rel_rowptr + u + 1) - __ldg(rel_rowptr + u);
        if (n_rel <= 0) {   // no ground truth: not counted; per-user values are NaN
            if (per_user != nullptr)
                for (int v = lane; v < n_cutoffs * kRmPerUser; v += 32)
                    per_user[row * n_cutoffs * kRmPerUser + v] = __longlong_as_double(0x7ff8000000000000ll);
            continue;
        }
        unsigned hit[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = 32 * j + lane;
            bool h = false;
            if (32 * j < k) {   // warp-uniform: the ballot below is reached by every lane
                if (r < k) {
                    const int32_t id = __ldg(ids + row * ld + r);
                    h = id >= 0 && id < n_items && excluded_item(rel_rowptr, rel_items, u, id);
                }
            }
            hit[j] = __ballot_sync(0xffffffffu, h);
        }
        // hits up to and including this lane's slot in each ballot word, and the first hit's rank
        int before = 0, first = 1 << 30;
        double ap_term[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool h = (hit[j] >> lane) & 1u;
            const int cum = before + __popc(hit[j] & (0xffffffffu >> (31 - lane)));
            ap_term[j] = h ? (double)cum / (double)(32 * j + lane + 1) : 0.0;
            if (first == (1 << 30) && hit[j]) first = 32 * j + __ffs(hit[j]) - 1;
            before += __popc(hit[j]);
        }
        for (int ci = 0; ci < n_cutoffs; ++ci) {
            const int c = cutoff[ci];
            const int ideal = (int64_t)c < n_rel ? c : (int)n_rel;
            int hits = 0;
            double dcg = 0.0, idcg = 0.0, ap = 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = 32 * j + lane;
                const int below = c - 32 * j;   // slots of word j that lie under the cutoff
                const unsigned m = below >= 32 ? 0xffffffffu : (below <= 0 ? 0u : (0xffffffffu >> (32 - below)));
                hits += __popc(hit[j] & m);
                if (r < c && ((hit[j] >> lane) & 1u)) dcg += w[j];
                if (r < ideal) idcg += w[j];
                if (r < c) ap += ap_term[j];
            }
            dcg = warp_sum(dcg);
            idcg = warp_sum(idcg);
            ap = warp_sum(ap);
            double val[kRmCols];
            val[0] = (double)hits / (double)c;
            val[1] = (double)hits / (double)n_rel;
            val[2] = first < c ? 1.0 : 0.0;
            val[3] = first < c ? 1.0 / (double)(first + 1) : 0.0;
            val[4] = dcg / idcg;
            val[5] = ap / (double)ideal;
            val[6] = 1.0;
#pragma unroll
            for (int m = 0; m < kRmCols; ++m) {
                const int v = ci * kRmCols + m;
                if ((v & 31) == lane) {
                    if (v < 32) acc0 += val[m]; else acc1 += val[m];
                }
            }
            if (per_user != nullptr && lane < kRmPerUser) {
                double out = val[0];
#pragma unroll
                for (int m = 1; m < kRmPerUser; ++m) out = lane == m ? val[m] : out;
                per_user[(row * n_cutoffs + ci) * kRmPerUser + lane] = out;
            }
        }
    }
    if (lane < n_vals) warp_acc[warp][lane] = acc0;
    if (lane + 32 < n_vals) warp_acc[warp][lane + 32] = acc1;
    __syncthreads();
    for (int v = threadIdx.x; v < n_vals; v += blockDim.x) {
        double s = warp_acc[0][v];
#pragma unroll
        for (int wi = 1; wi < kRmWarps; ++wi) s += warp_acc[wi][v];
        partials[(int64_t)v * gridDim.x + blockIdx.x] = s;
    }
}

// one block per value: thread t adds partials t, t + 256, ... in order, then a fixed shared-memory tree
__global__ void __launch_bounds__(kRmReduceThreads) rank_metrics_reduce_kernel(const double *__restrict__ partials,
                                                                              int64_t n_blocks, double *__restrict__ sums) {
    __shared__ double sh[kRmReduceThreads];
    const double *p = partials + (int64_t)blockIdx.x * n_blocks;
    double s = 0.0;
    for (int64_t b = threadIdx.x; b < n_blocks; b += kRmReduceThreads) s += p[b];
    sh[threadIdx.x] = s;
    __syncthreads();
#pragma unroll
    for (int o = kRmReduceThreads / 2; o; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[blockIdx.x] = sh[0];
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_rank_metrics_workspace_bytes(int64_t n_rows, int32_t n_cutoffs) {
    if (n_rows <= 0 || n_cutoffs <= 0) return 0;
    return align_up((size_t)cdiv(n_rows, kRmRowsPerBlock) * (size_t)n_cutoffs * kRmCols * sizeof(double));
}

extern "C" int cbrs_rank_metrics(const int32_t *ids, int64_t ld, int64_t n_rows, int32_t k, int32_t n_items,
                                 const int64_t *users, int64_t n_users, const int64_t *rel_rowptr,
                                 const int32_t *rel_items, const int32_t *cutoffs_host, int32_t n_cutoffs,
                                 double *sums_out, double *per_user_out, void *workspace, size_t workspace_bytes,
                                 void *stream) {
    CBRS_REQUIRE(!rel_rowptr == !rel_items, CBRS_E_INVALID, "rank_metrics: %s is null but %s is not",
                 rel_rowptr ? "rel_items" : "rel_rowptr", rel_rowptr ? "rel_rowptr" : "rel_items");
    CBRS_REQUIRE(k >= 1 && k <= 128, CBRS_E_INVALID, "rank_metrics: k=%d outside [1, 128]", k);
    CBRS_REQUIRE(n_cutoffs >= 1 && n_cutoffs <= kRmMaxCutoffs && cutoffs_host, CBRS_E_INVALID,
                 "rank_metrics: n_cutoffs=%d outside [1, %d] (or null cutoffs)", n_cutoffs, kRmMaxCutoffs);
    Cutoffs cut = {};
    for (int i = 0; i < n_cutoffs; ++i) {
        cut.c[i] = cutoffs_host[i];
        CBRS_REQUIRE(cut.c[i] >= 1 && cut.c[i] <= k, CBRS_E_INVALID, "rank_metrics: cutoff %d outside [1, k=%d]",
                     cut.c[i], k);
        CBRS_REQUIRE(i == 0 || cut.c[i] > cut.c[i - 1], CBRS_E_INVALID,
                     "rank_metrics: cutoffs not strictly ascending (%d after %d)", cut.c[i], cut.c[i - 1]);
    }
    CBRS_REQUIRE(n_rows >= 0 && n_items >= 0 && n_users >= 0 && sums_out && (n_rows == 0 || (ids && ld >= k)),
                 CBRS_E_INVALID, "rank_metrics: n_rows=%lld ld=%lld k=%d n_items=%d n_users=%lld (or null ids / sums)",
                 (long long)n_rows, (long long)ld, k, n_items, (long long)n_users);
    cudaStream_t s = (cudaStream_t)stream;
    const int n_vals = n_cutoffs * kRmCols;
    if (n_rows == 0) {
        const cudaError_t e = cudaMemsetAsync(sums_out, 0, (size_t)n_vals * sizeof(double), s);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "rank_metrics: %s", cudaGetErrorString(e));
        return CBRS_OK;
    }
    const int64_t n_blocks = cdiv(n_rows, kRmRowsPerBlock);
    CBRS_REQUIRE(n_blocks < (1ll << 31), CBRS_E_INVALID, "rank_metrics: n_rows=%lld too large", (long long)n_rows);
    CBRS_REQUIRE(workspace && workspace_bytes >= cbrs_rank_metrics_workspace_bytes(n_rows, n_cutoffs), CBRS_E_WORKSPACE,
                 "rank_metrics: workspace of %zu bytes, %zu needed", workspace_bytes,
                 cbrs_rank_metrics_workspace_bytes(n_rows, n_cutoffs));
    double *partials = (double *)workspace;
    rank_metrics_kernel<<<(unsigned)n_blocks, kRmWarps * 32, 0, s>>>(ids, ld, n_rows, k, n_items, users, n_users,
                                                                     rel_rowptr, rel_items, cut, n_cutoffs,
                                                                     per_user_out, partials);
    CBRS_CHECK_LAUNCH("rank_metrics");
    rank_metrics_reduce_kernel<<<(unsigned)n_vals, kRmReduceThreads, 0, s>>>(partials, n_blocks, sums_out);
    CBRS_CHECK_LAUNCH("rank_metrics_reduce");
    return CBRS_OK;
}
