// Backward of the fused GAT layer (csrc/gat.cu) for the training step, scope row (f)-1.
//
// Forward (SURVEY.md Appendix A.4, spektral GATConv as built at
// /root/reference/src/models/gnn.py:321-328): edge set E = {raw A minus self loops} + {(i,i)};
//   s_ij = p_i + q_j,  e_ij = leaky_relu_0.2(s_ij),  m_i = max_j e_ij,  w_ij = exp(e_ij - m_i),
//   S_i = sum_j w_ij + 1e-9,  alpha_ij = w_ij / S_i,  o_i = sum_j alpha_ij z_j,  y_i = act(o_i + b).
// Given dO = dY * act'(y):
//   dalpha_ij = dO_i . z_j                t_i = sum_j alpha_ij dalpha_ij = dO_i . o_i
//   de_ij = alpha_ij (dalpha_ij - t_i)    ds_ij = de_ij * (s_ij > 0 ? 1 : 0.2)
//   dp_i = sum_j ds_ij        dq_j = sum_i ds_ij        dz_j = sum_i alpha_ij dO_i
// (the max shift carries no gradient up to the 1e-9 term; TensorFlow's autograd result differs by
// O(1e-9 / S_i), below float32 resolution of the sums).
//
// dq and dz are sums over the edges that END in j.  Every adjacency of the reference is symmetrised
// (config.yaml:36, src/utilities/math.py:13-20), duplicates included, so the edges ending in j are the
// transposes of row j's own list: both passes are row gathers over the same CSR, no transposed
// structure, no atomics, fixed summation order.
//   gat_bwd_stats : per row m_i, S_i (recomputed, 8 B per node instead of saving alpha per edge), t_i
//   gat_bwd_rows  : pass A (dp_i) and pass B (dq_j, dz_j) in one kernel, one warp per row
#include "common.cuh"

namespace cbrs {

struct GatBwdParams {
    const int64_t *rowptr;
    const int32_t *colidx;
    int64_t n_rows;
    const float *z; int64_t ldz;
    const float *p; const float *q;
    const float *y; int64_t ldy;      // forward output (post activation)
    const float *bias;
    const float *d_o; int64_t ldo;    // dO = dY * act'(y)
    int32_t h;
    float *m; float *s; float *t;     // [N] each
    float *dp; float *dq;             // [N]
    float *dz; int64_t lddz;          // [N, h]
};

__device__ __forceinline__ float lrelu02(float x) { return x > 0.f ? x : 0.2f * x; }
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(256) gat_bwd_stats_kernel(const GatBwdParams p) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= p.n_rows) return;
    const int64_t b = p.rowptr[row], e = p.rowptr[row + 1];
    const float pi = p.p[row];
    float m = lrelu02(pi + p.q[row]);  // the self edge
    for (int64_t k = b + lane; k < e; k += 32) {
        const int c = p.colidx[k];
        if (c != row) m = fmaxf(m, lrelu02(pi + p.q[c]));
    }
    m = warp_max(m);
    float s = 0.f;
    for (int64_t k = b + lane; k < e; k += 32) {
        const int c = p.colidx[k];
        if (c != row) s += expf(lrelu02(pi + p.q[c]) - m);
    }
    s = warp_sum(s) + expf(lrelu02(pi + p.q[row]) - m);
    float t = 0.f;
    for (int c = lane; c < p.h; c += 32) {
        const float g = p.d_o[row * p.ldo + c];
        if (g != 0.f) t = fmaf(g, p.y[row * p.ldy + c] - (p.bias ? p.bias[c] : 0.f), t);
    }
    t = warp_sum(t);
    if (lane == 0) {
        p.m[row] = m;
        p.s[row] = s + 1e-9f;
        p.t[row] = t;
    }
}

// dot of two h-wide rows, read by ONE lane
__device__ __forceinline__ float row_dot(const float *a, const float *b, int h, bool vec4) {
    float acc = 0.f;
    if (vec4) {
        for (int c = 0; c < h; c += 4) {
            const float4 x = *reinterpret_cast<const float4 *>(a + c);
            const float4 y = *reinterpret_cast<const float4 *>(b + c);
            acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
        }
    } else {
        for (int c = 0; c < h; ++c) acc = fmaf(a[c], b[c], acc);
    }
    return acc;
}

constexpr int kGatBwdMaxAcc = 8;  // h <= 256

__global__ void __launch_bounds__(256) gat_bwd_rows_kernel(const GatBwdParams p, int vec4) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= p.n_rows) return;
    const int64_t b = p.rowptr[row], e = p.rowptr[row + 1];
    const int64_t n_edges = e - b + 1;  // + the self edge, taken as the last one
    const float p_r = p.p[row], q_r = p.q[row];
    const float m_r = p.m[row], s_r = p.s[row], t_r = p.t[row];
    const float *do_r = p.d_o + row * p.ldo;
    const float *z_r = p.z + row * p.ldz;
    float dp_lane = 0.f, dq_lane = 0.f;
    float acc[kGatBwdMaxAcc];
#pragma unroll
    for (int k = 0; k < kGatBwdMaxAcc; ++k) acc[k] = 0.f;
    for (int64_t base = 0; base < n_edges; base += 32) {
        const int64_t k = base + lane;
        int c = -1;
        float coef = 0.f;  // alpha of the edge that ends in `row` and starts in c
        if (k < n_edges) {
            c = k < n_edges - 1 ? p.colidx[b + k] : (int)row;
            if (k < n_edges - 1 && c == row) c = -1;  // existing self loops are replaced by the one added above
        }
        if (c >= 0) {
            // pass A: edge (row -> c): row attends to c
            const float s_a = p_r + p.q[c];
            const float alpha_a = expf(lrelu02(s_a) - m_r) / s_r;
            const float dal_a = row_dot(do_r, p.z + (int64_t)c * p.ldz, p.h, vec4);
            dp_lane += alpha_a * (dal_a - t_r) * (s_a > 0.f ? 1.f : 0.2f);
            // pass B: edge (c -> row): c attends to row
            const float s_b = p.p[c] + q_r;
            coef = expf(lrelu02(s_b) - p.m[c]) / p.s[c];
            const float dal_b = row_dot(p.d_o + (int64_t)c * p.ldo, z_r, p.h, vec4);
            dq_lane += coef * (dal_b - p.t[c]) * (s_b > 0.f ? 1.f : 0.2f);
        }
        const int cnt = n_edges - base < 32 ? (int)(n_edges - base) : 32;
        for (int u = 0; u < cnt; ++u) {
            const int cu = __shfl_sync(0xffffffffu, c, u);
            const float au = __shfl_sync(0xffffffffu, coef, u);
            if (cu < 0) continue;
            const float *src = p.d_o + (int64_t)cu * p.ldo;
#pragma unroll
            for (int k2 = 0; k2 < kGatBwdMaxAcc; ++k2) {
                const int col = lane + 32 * k2;
                if (col < p.h) acc[k2] = fmaf(au, src[col], acc[k2]);
            }
        }
    }
    dp_lane = warp_sum(dp_lane);
    dq_lane = warp_sum(dq_lane);
    if (lane == 0) {
        p.dp[row] = dp_lane;
        p.dq[row] = dq_lane;
    }
#pragma unroll
    for (int k2 = 0; k2 < kGatBwdMaxAcc; ++k2) {
        const int col = lane + 32 * k2;
        if (col < p.h) p.dz[row * p.lddz + col] = acc[k2];
    }
}

// dz += dp (x) a_self + dq (x) a_neigh   (p = z . a_self, q = z . a_neigh)
__global__ void gat_bwd_combine_kernel(float *__restrict__ dz, int64_t lddz, const float *__restrict__ dp,
                                       const float *__restrict__ dq, const float *__restrict__ a_self,
                                       const float *__restrict__ a_neigh, int64_t n_rows, int32_t h) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * h) return;
    const int64_t r = i / h;
    const int c = (int)(i % h);
    dz[r * lddz + c] = fmaf(dq[r], a_neigh[c], fmaf(dp[r], a_self[c], dz[r * lddz + c]));
}

// ---- row-slice form for the row partition (cbrs_gat_backward_stats_rows / cbrs_gat_backward_grad_rows) ----------
// The same per-row arithmetic as the two kernels above, on rows [row_offset, row_offset + n_rows) of a graph whose
// column ids are global, so every output row has the bits of the whole-graph call.  Inputs are whole-graph arrays read
// at global rows; outputs are views of the slice's rows (as in cbrs_gat_csr).  The stats live in a caller-owned [N, 3]
// array (m, S, t) instead of the workspace: the rows phase reads the stats of neighbour rows, which another rank
// computed and stored into this rank's copy.  The combine (dz += dp a_self + dq a_neigh) is folded into the rows
// kernel's epilogue with the operand order of gat_bwd_combine_kernel, so no kernel reads back an output (an output may
// be a multicast address).
struct GatBwdSliceParams {
    const int64_t *rowptr;
    const int32_t *colidx;
    int64_t n_rows, row_offset;
    const float *z; int64_t ldz;
    const float *p; const float *q;
    const float *y; int64_t ldy;
    const float *bias;
    const float *d_o; int64_t ldo;
    int32_t h;
    const float *stats_in;            // [N, 3], read by the rows phase
    float *stats;                     // [n_rows, 3], written by the stats phase
    const float *a_self; const float *a_neigh;
    float *dp; float *dq;             // [n_rows]
    float *dz; int64_t lddz;          // [n_rows, h]
    float *stats_peer[CBRS_MAX_PEERS - 1];
    float *dp_peer[CBRS_MAX_PEERS - 1];
    float *dq_peer[CBRS_MAX_PEERS - 1];
    float *dz_peer[CBRS_MAX_PEERS - 1];
    int n_peer;
};

__global__ void __launch_bounds__(256) gat_bwd_stats_slice_kernel(const GatBwdSliceParams p) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= p.n_rows) return;
    const int64_t g = row + p.row_offset;
    const int64_t b = p.rowptr[row], e = p.rowptr[row + 1];
    const float pi = p.p[g];
    float m = lrelu02(pi + p.q[g]);
    for (int64_t k = b + lane; k < e; k += 32) {
        const int c = p.colidx[k];
        if (c != g) m = fmaxf(m, lrelu02(pi + p.q[c]));
    }
    m = warp_max(m);
    float s = 0.f;
    for (int64_t k = b + lane; k < e; k += 32) {
        const int c = p.colidx[k];
        if (c != g) s += expf(lrelu02(pi + p.q[c]) - m);
    }
    s = warp_sum(s) + expf(lrelu02(pi + p.q[g]) - m);
    float t = 0.f;
    for (int c = lane; c < p.h; c += 32) {
        const float gr = p.d_o[g * p.ldo + c];
        if (gr != 0.f) t = fmaf(gr, p.y[g * p.ldy + c] - (p.bias ? p.bias[c] : 0.f), t);
    }
    t = warp_sum(t);
    if (lane < 3) {
        const float v = lane == 0 ? m : (lane == 1 ? s + 1e-9f : t);
        p.stats[row * 3 + lane] = v;
        for (int r = 0; r < p.n_peer; ++r) p.stats_peer[r][row * 3 + lane] = v;
    }
}

__global__ void __launch_bounds__(256) gat_bwd_rows_slice_kernel(const GatBwdSliceParams p, int vec4) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= p.n_rows) return;
    const int64_t g = row + p.row_offset;
    const int64_t b = p.rowptr[row], e = p.rowptr[row + 1];
    const int64_t n_edges = e - b + 1;
    const float p_r = p.p[g], q_r = p.q[g];
    const float m_r = p.stats_in[g * 3], s_r = p.stats_in[g * 3 + 1], t_r = p.stats_in[g * 3 + 2];
    const float *do_r = p.d_o + g * p.ldo;
    const float *z_r = p.z + g * p.ldz;
    float dp_lane = 0.f, dq_lane = 0.f;
    float acc[kGatBwdMaxAcc];
#pragma unroll
    for (int k = 0; k < kGatBwdMaxAcc; ++k) acc[k] = 0.f;
    for (int64_t base = 0; base < n_edges; base += 32) {
        const int64_t k = base + lane;
        int c = -1;
        float coef = 0.f;
        if (k < n_edges) {
            c = k < n_edges - 1 ? p.colidx[b + k] : (int)g;
            if (k < n_edges - 1 && c == g) c = -1;
        }
        if (c >= 0) {
            const float s_a = p_r + p.q[c];
            const float alpha_a = expf(lrelu02(s_a) - m_r) / s_r;
            const float dal_a = row_dot(do_r, p.z + (int64_t)c * p.ldz, p.h, vec4);
            dp_lane += alpha_a * (dal_a - t_r) * (s_a > 0.f ? 1.f : 0.2f);
            const float s_b = p.p[c] + q_r;
            coef = expf(lrelu02(s_b) - p.stats_in[(int64_t)c * 3]) / p.stats_in[(int64_t)c * 3 + 1];
            const float dal_b = row_dot(p.d_o + (int64_t)c * p.ldo, z_r, p.h, vec4);
            dq_lane += coef * (dal_b - p.stats_in[(int64_t)c * 3 + 2]) * (s_b > 0.f ? 1.f : 0.2f);
        }
        const int cnt = n_edges - base < 32 ? (int)(n_edges - base) : 32;
        for (int u = 0; u < cnt; ++u) {
            const int cu = __shfl_sync(0xffffffffu, c, u);
            const float au = __shfl_sync(0xffffffffu, coef, u);
            if (cu < 0) continue;
            const float *src = p.d_o + (int64_t)cu * p.ldo;
#pragma unroll
            for (int k2 = 0; k2 < kGatBwdMaxAcc; ++k2) {
                const int col = lane + 32 * k2;
                if (col < p.h) acc[k2] = fmaf(au, src[col], acc[k2]);
            }
        }
    }
    // the xor butterfly leaves the same sum in every lane, so each lane can apply the combine itself
    dp_lane = warp_sum(dp_lane);
    dq_lane = warp_sum(dq_lane);
    if (lane == 0) {
        p.dp[row] = dp_lane;
        p.dq[row] = dq_lane;
        for (int r = 0; r < p.n_peer; ++r) {
            p.dp_peer[r][row] = dp_lane;
            p.dq_peer[r][row] = dq_lane;
        }
    }
#pragma unroll
    for (int k2 = 0; k2 < kGatBwdMaxAcc; ++k2) {
        const int col = lane + 32 * k2;
        if (col < p.h) {
            const float v = fmaf(dq_lane, p.a_neigh[col], fmaf(dp_lane, p.a_self[col], acc[k2]));
            p.dz[row * p.lddz + col] = v;
            for (int r = 0; r < p.n_peer; ++r) p.dz_peer[r][row * p.lddz + col] = v;
        }
    }
}

}  // namespace cbrs

using namespace cbrs;

// copies a host list of n peer addresses into dst[CBRS_MAX_PEERS - 1]; false when the list or an entry is null
static bool take_peers(float **dst, void *const *host, int n) {
    for (int r = 0; r < CBRS_MAX_PEERS - 1; ++r) dst[r] = nullptr;
    if (n > 0 && !host) return false;
    for (int r = 0; r < n; ++r) {
        dst[r] = (float *)host[r];
        if (!dst[r]) return false;
    }
    return true;
}

extern "C" int cbrs_gat_backward_stats_rows(const cbrs_csr_t *g, int64_t row_offset, const float *pvec,
                                            const float *qvec, const float *y, int64_t ldy, const float *bias,
                                            const float *d_o, int64_t ldo, int32_t h, float *stats,
                                            void *const *stats_peers_host, int n_peers, void *stream) {
    CBRS_REQUIRE(g && pvec && qvec && y && d_o && stats, CBRS_E_INVALID, "gat_backward_stats_rows: null argument");
    CBRS_REQUIRE(h > 0 && ldy >= h && ldo >= h && row_offset >= 0, CBRS_E_INVALID,
                 "gat_backward_stats_rows: h=%d ldy=%lld ldo=%lld row_offset=%lld", h, (long long)ldy, (long long)ldo,
                 (long long)row_offset);
    CBRS_REQUIRE(n_peers >= 0 && n_peers < CBRS_MAX_PEERS, CBRS_E_INVALID,
                 "gat_backward_stats_rows: n_peers=%d (at most %d peer copies)", n_peers, CBRS_MAX_PEERS - 1);
    CBRS_REQUIRE(g->n_rows >= 0 && (g->n_rows == 0 || g->rowptr) && (g->nnz == 0 || g->colidx), CBRS_E_INVALID,
                 "gat_backward_stats_rows: bad graph descriptor");
    GatBwdSliceParams p = {};
    CBRS_REQUIRE(take_peers(p.stats_peer, stats_peers_host, n_peers), CBRS_E_INVALID,
                 "gat_backward_stats_rows: null peer copy");
    if (g->n_rows == 0) return CBRS_OK;
    p.rowptr = g->rowptr; p.colidx = g->colidx; p.n_rows = g->n_rows; p.row_offset = row_offset;
    p.p = pvec; p.q = qvec; p.y = y; p.ldy = ldy; p.bias = bias; p.d_o = d_o; p.ldo = ldo; p.h = h;
    p.stats = stats; p.n_peer = n_peers;
    gat_bwd_stats_slice_kernel<<<(unsigned)cdiv(g->n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(p);
    CBRS_CHECK_LAUNCH("gat_bwd_stats_slice");
    return CBRS_OK;
}

extern "C" int cbrs_gat_backward_grad_rows(const cbrs_csr_t *g, int64_t row_offset, const float *z, int64_t ldz,
                                           const float *pvec, const float *qvec, const float *d_o, int64_t ldo,
                                           int32_t h, const float *stats, const float *a_self, const float *a_neigh,
                                           float *dz, int64_t lddz, float *dp, float *dq, void *const *dz_peers_host,
                                           void *const *dp_peers_host, void *const *dq_peers_host, int n_peers,
                                           void *stream) {
    CBRS_REQUIRE(g && z && pvec && qvec && d_o && stats && a_self && a_neigh && dz && dp && dq, CBRS_E_INVALID,
                 "gat_backward_grad_rows: null argument");
    CBRS_REQUIRE(h > 0 && h <= 32 * kGatBwdMaxAcc && ldz >= h && ldo >= h && lddz >= h && row_offset >= 0,
                 CBRS_E_INVALID, "gat_backward_grad_rows: h=%d (max %d), a leading dimension or row_offset is bad", h,
                 32 * kGatBwdMaxAcc);
    CBRS_REQUIRE(n_peers >= 0 && n_peers < CBRS_MAX_PEERS, CBRS_E_INVALID,
                 "gat_backward_grad_rows: n_peers=%d (at most %d peer copies)", n_peers, CBRS_MAX_PEERS - 1);
    CBRS_REQUIRE(g->n_rows >= 0 && (g->n_rows == 0 || g->rowptr) && (g->nnz == 0 || g->colidx), CBRS_E_INVALID,
                 "gat_backward_grad_rows: bad graph descriptor");
    GatBwdSliceParams p = {};
    CBRS_REQUIRE(take_peers(p.dz_peer, dz_peers_host, n_peers) && take_peers(p.dp_peer, dp_peers_host, n_peers) &&
                     take_peers(p.dq_peer, dq_peers_host, n_peers),
                 CBRS_E_INVALID, "gat_backward_grad_rows: null peer copy");
    if (g->n_rows == 0) return CBRS_OK;
    p.rowptr = g->rowptr; p.colidx = g->colidx; p.n_rows = g->n_rows; p.row_offset = row_offset;
    p.z = z; p.ldz = ldz; p.p = pvec; p.q = qvec; p.d_o = d_o; p.ldo = ldo; p.h = h; p.stats_in = stats;
    p.a_self = a_self; p.a_neigh = a_neigh; p.dz = dz; p.lddz = lddz; p.dp = dp; p.dq = dq; p.n_peer = n_peers;
    const int vec4 = (h % 4 == 0) && (ldz % 4 == 0) && (ldo % 4 == 0) && ((uintptr_t)z % 16 == 0) && ((uintptr_t)d_o % 16 == 0);
    gat_bwd_rows_slice_kernel<<<(unsigned)cdiv(g->n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(p, vec4);
    CBRS_CHECK_LAUNCH("gat_bwd_rows_slice");
    return CBRS_OK;
}

extern "C" size_t cbrs_gat_backward_workspace_bytes(int64_t n_rows) {
    return 3 * align_up((size_t)n_rows * sizeof(float)) + 256;
}

extern "C" int cbrs_gat_backward(const cbrs_csr_t *g, const float *z, int64_t ldz, const float *pvec, const float *qvec,
                                 const float *y, int64_t ldy, const float *bias, const float *d_o, int64_t ldo, int32_t h,
                                 const float *a_self, const float *a_neigh, float *dz, int64_t lddz, float *dp, float *dq,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(g && z && pvec && qvec && y && d_o && a_self && a_neigh && dz && dp && dq, CBRS_E_INVALID,
                 "gat_backward: null argument");
    CBRS_REQUIRE(h > 0 && h <= 32 * kGatBwdMaxAcc && ldz >= h && ldy >= h && ldo >= h && lddz >= h, CBRS_E_INVALID,
                 "gat_backward: h=%d (max %d) or a leading dimension is too small", h, 32 * kGatBwdMaxAcc);
    CBRS_REQUIRE(g->n_rows >= 0 && (g->n_rows == 0 || g->rowptr) && (g->nnz == 0 || g->colidx), CBRS_E_INVALID,
                 "gat_backward: bad graph descriptor");
    if (g->n_rows == 0) return CBRS_OK;
    CBRS_REQUIRE(workspace && workspace_bytes >= cbrs_gat_backward_workspace_bytes(g->n_rows), CBRS_E_WORKSPACE,
                 "gat_backward: workspace too small");
    Arena a(workspace, workspace_bytes);
    GatBwdParams p;
    p.rowptr = g->rowptr; p.colidx = g->colidx; p.n_rows = g->n_rows;
    p.z = z; p.ldz = ldz; p.p = pvec; p.q = qvec; p.y = y; p.ldy = ldy; p.bias = bias; p.d_o = d_o; p.ldo = ldo; p.h = h;
    p.m = a.take<float>((size_t)g->n_rows); p.s = a.take<float>((size_t)g->n_rows); p.t = a.take<float>((size_t)g->n_rows);
    p.dp = dp; p.dq = dq; p.dz = dz; p.lddz = lddz;
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned grid = (unsigned)cdiv(g->n_rows * 32, 256);
    gat_bwd_stats_kernel<<<grid, 256, 0, s>>>(p);
    CBRS_CHECK_LAUNCH("gat_bwd_stats");
    const int vec4 = (h % 4 == 0) && (ldz % 4 == 0) && (ldo % 4 == 0) && ((uintptr_t)z % 16 == 0) && ((uintptr_t)d_o % 16 == 0);
    gat_bwd_rows_kernel<<<grid, 256, 0, s>>>(p, vec4);
    CBRS_CHECK_LAUNCH("gat_bwd_rows");
    gat_bwd_combine_kernel<<<(unsigned)cdiv(g->n_rows * h, 256), 256, 0, s>>>(dz, lddz, dp, dq, a_self, a_neigh, g->n_rows, h);
    CBRS_CHECK_LAUNCH("gat_bwd_combine");
    return CBRS_OK;
}
