// CSR x dense propagation kernels for sm_100a: weighted SpMM (GCN / LightGCN),
// sum and mean aggregators (GraphSAGE).  Rows P1, P2 (aggregate), P4.
//
// Replaces tf.sparse.sparse_dense_matmul reached through spektral GCNConv and
// ops.modal_dot (/root/reference/src/layers/lightgcn_conv.py:53) and the
// gather + unsorted_segment_mean of GraphSageConv (built at src/models/gnn.py:354-361).
//
// HBM-bound gather: per edge 8 B of (col,val) stream + one D*4-byte feature row.
//  * G lanes own one chunk of a row; lane l holds 4 consecutive floats (one
//    128-bit load per edge per lane), so a 128-wide row is one 512-B warp request;
//  * (col,val) are fetched G at a time, coalesced, L1::no_allocate, and handed
//    round with shuffles; 8 independent row loads are in flight per group;
//  * accumulation order inside a chunk is ascending column == the oracle's;
//  * rows longer than chunk_edges are split: each chunk parks a partial and a
//    second kernel adds the partials in ascending chunk order (fixed tree).
#include "common.cuh"

#include <cuda_bf16.h>

#include <type_traits>

namespace cbrs {

struct SpmmParams {
    const int64_t *rowptr;
    const int32_t *colidx;
    const float *vals;
    const int32_t *chunk_row;
    const int64_t *chunk_begin;
    const int32_t *chunk_slot;
    const int32_t *chunk_len;  // explicit chunk lengths (column-blocked decomposition) or null
    int64_t n_chunks;
    int32_t chunk_edges;
    const void *x;  // float32, or bf16 when the kernel is instantiated with XT = __nv_bfloat16
    int64_t ldx;
    float *y;
    int64_t ldy;
    int32_t d;
    int agg;
    const float *bias;
    int relu;
    float *partial;  // [n_slots, d]
    const int32_t *heavy_row;
    const int64_t *heavy_slot_ptr;
    int64_t n_heavy;
    // multi-GPU: every finished row is also stored into these peer-mapped copies of y (NVLink)
    float *y_peer[CBRS_MAX_PEERS - 1];
    int n_peer;
};

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    float4 v;
    __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ void load(const float *p) { v = ldg4(p); }
    __device__ __forceinline__ void load_plain(const float *p) { v = *reinterpret_cast<const float4 *>(p); }
    // 4 bf16 (8 bytes) -> 4 floats; the conversion is exact (bf16 is the top half of a float)
    __device__ __forceinline__ void load(const __nv_bfloat16 *p) {
        const uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
        v = make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                        __uint_as_float(r.y & 0xffff0000u));
    }
    __device__ __forceinline__ void fma(float a, const Vec &x) {
        v.x = fmaf(a, x.v.x, v.x); v.y = fmaf(a, x.v.y, v.y); v.z = fmaf(a, x.v.z, v.z); v.w = fmaf(a, x.v.w, v.w);
    }
    __device__ __forceinline__ void add(const Vec &x) { v.x += x.v.x; v.y += x.v.y; v.z += x.v.z; v.w += x.v.w; }
    __device__ __forceinline__ void div(float c) { v.x /= c; v.y /= c; v.z /= c; v.w /= c; }
    __device__ __forceinline__ void epilogue(const float *bias, int relu) {
        if (bias) { float4 b = ldg4(bias); v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w; }
        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    }
    __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float4 *>(p) = v; }
};
template <>
struct Vec<1> {
    float v;
    __device__ __forceinline__ void zero() { v = 0.f; }
    __device__ __forceinline__ void load(const float *p) { v = __ldg(p); }
    __device__ __forceinline__ void load_plain(const float *p) { v = *p; }
    __device__ __forceinline__ void load(const __nv_bfloat16 *p) {
        v = __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short *>(p)) << 16);
    }
    __device__ __forceinline__ void fma(float a, const Vec &x) { v = fmaf(a, x.v, v); }
    __device__ __forceinline__ void add(const Vec &x) { v += x.v; }
    __device__ __forceinline__ void div(float c) { v /= c; }
    __device__ __forceinline__ void epilogue(const float *bias, int relu) {
        if (bias) v += __ldg(bias);
        if (relu) v = fmaxf(v, 0.f);
    }
    __device__ __forceinline__ void store(float *p) const { *p = v; }
};

// 8-wide lane slice: used for bf16 rows, where 8 elements are one 16-byte load and a 128-wide row needs only 16
// lanes - two chunks share a warp and every instruction of the edge loop serves two edges
template <>
struct Vec<8> {
    float4 a, b;
    __device__ __forceinline__ void zero() { a = make_float4(0.f, 0.f, 0.f, 0.f); b = a; }
    __device__ __forceinline__ void load_plain(const float *p) {
        a = *reinterpret_cast<const float4 *>(p); b = *reinterpret_cast<const float4 *>(p + 4);
    }
    __device__ __forceinline__ void from_raw(const uint4 r) {
        a = make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                        __uint_as_float(r.y & 0xffff0000u));
        b = make_float4(__uint_as_float(r.z << 16), __uint_as_float(r.z & 0xffff0000u), __uint_as_float(r.w << 16),
                        __uint_as_float(r.w & 0xffff0000u));
    }
    __device__ __forceinline__ void load(const __nv_bfloat16 *p) { from_raw(__ldg(reinterpret_cast<const uint4 *>(p))); }
    __device__ __forceinline__ void fma(float s, const Vec &x) {
        a.x = fmaf(s, x.a.x, a.x); a.y = fmaf(s, x.a.y, a.y); a.z = fmaf(s, x.a.z, a.z); a.w = fmaf(s, x.a.w, a.w);
        b.x = fmaf(s, x.b.x, b.x); b.y = fmaf(s, x.b.y, b.y); b.z = fmaf(s, x.b.z, b.z); b.w = fmaf(s, x.b.w, b.w);
    }
    __device__ __forceinline__ void add(const Vec &x) {
        a.x += x.a.x; a.y += x.a.y; a.z += x.a.z; a.w += x.a.w; b.x += x.b.x; b.y += x.b.y; b.z += x.b.z; b.w += x.b.w;
    }
    __device__ __forceinline__ void div(float c) {
        a.x /= c; a.y /= c; a.z /= c; a.w /= c; b.x /= c; b.y /= c; b.z /= c; b.w /= c;
    }
    __device__ __forceinline__ void epilogue(const float *bias, int relu) {
        if (bias) {
            const float4 u = ldg4(bias), v = ldg4(bias + 4);
            a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w; b.x += v.x; b.y += v.y; b.z += v.z; b.w += v.w;
        }
        if (relu) {
            a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
            b.x = fmaxf(b.x, 0.f); b.y = fmaxf(b.y, 0.f); b.z = fmaxf(b.z, 0.f); b.w = fmaxf(b.w, 0.f);
        }
    }
    __device__ __forceinline__ void store(float *p) const {
        *reinterpret_cast<float4 *>(p) = a; *reinterpret_cast<float4 *>(p + 4) = b;
    }
};

constexpr int kSpmmThreads = 256;

template <int G, int VEC, int UMAX = 4, int MINB = 4, typename XT = float>
__global__ void __launch_bounds__(kSpmmThreads, MINB) spmm_chunk_kernel(const SpmmParams p) {
    constexpr int U = G < UMAX ? G : UMAX;  // independent row loads in flight per group
    const int64_t gid = ((int64_t)blockIdx.x * kSpmmThreads + threadIdx.x) / G;
    if (gid >= p.n_chunks) return;
    const int lane = threadIdx.x & 31;
    const int lg = lane & (G - 1);
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));

    const int32_t row = p.chunk_row[gid];
    const int64_t row_b = p.rowptr[row], row_e = p.rowptr[row + 1];
    const int64_t b = p.chunk_begin[gid];
    const int64_t e = p.chunk_len ? b + p.chunk_len[gid] : ((b + p.chunk_edges < row_e) ? b + p.chunk_edges : row_e);
    const int32_t slot = p.chunk_slot[gid];
    const bool weighted = (p.agg == CBRS_AGG_WEIGHTED) && p.vals != nullptr;
    // row stride in bytes as a 32-bit value (checked on the host): a row address is one IMAD.WIDE per edge
    const int ldx_bytes = (int)(p.ldx * (int64_t)sizeof(XT));

    for (int c0 = 0; c0 < p.d; c0 += G * VEC) {
        const int col = c0 + lg * VEC;
        const bool col_ok = col < p.d;
        const char *xcol = reinterpret_cast<const char *>(reinterpret_cast<const XT *>(p.x) + (col_ok ? col : 0));
        Vec<VEC> acc;
        acc.zero();
        // (col,val) of the next G edges are fetched while the current G rows are in flight
        int c_next = 0;
        float v_next = 0.f;
        if (b + lg < e) {
            c_next = ld_stream_i32(p.colidx + b + lg);
            v_next = weighted ? ld_stream_f32(p.vals + b + lg) : 1.f;
        }
        for (int64_t base = b; base < e; base += G) {
            const int c = c_next;
            const float v = v_next;
            const int64_t nidx = base + G + lg;
            c_next = 0;
            v_next = 0.f;
            if (nidx < e) {
                c_next = ld_stream_i32(p.colidx + nidx);
                v_next = weighted ? ld_stream_f32(p.vals + nidx) : 1.f;
            }
            const int cnt = (e - base < G) ? (int)(e - base) : G;
#pragma unroll
            for (int k0 = 0; k0 < G; k0 += U) {
                if (k0 >= cnt) break;
                int cc[U];
                float vv[U];
                Vec<VEC> xr[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    cc[u] = __shfl_sync(gmask, c, k0 + u, G);
                    vv[u] = __shfl_sync(gmask, v, k0 + u, G);
                }
                if constexpr (!std::is_same<XT, float>::value && VEC == 4) {
                    // bf16 rows: keep the raw 8-byte loads in flight (2 registers each) and widen at the FMA, so twice
                    // as many row loads fit in the register budget - the same BYTES in flight per warp as the fp32 kernel
                    uint2 raw[U];
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt)
                            raw[u] = __ldg(reinterpret_cast<const uint2 *>(xcol + (int64_t)cc[u] * ldx_bytes));
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt) {
                            xr[0].v = make_float4(__uint_as_float(raw[u].x << 16), __uint_as_float(raw[u].x & 0xffff0000u),
                                                  __uint_as_float(raw[u].y << 16), __uint_as_float(raw[u].y & 0xffff0000u));
                            acc.fma(vv[u], xr[0]);
                        }
                } else if constexpr (!std::is_same<XT, float>::value && VEC == 8) {
                    uint4 raw[U];
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt)
                            raw[u] = __ldg(reinterpret_cast<const uint4 *>(xcol + (int64_t)cc[u] * ldx_bytes));
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt) {
                            xr[0].from_raw(raw[u]);
                            acc.fma(vv[u], xr[0]);
                        }
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt)
                            xr[u].load(reinterpret_cast<const XT *>(xcol + (int64_t)cc[u] * ldx_bytes));
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (col_ok && k0 + u < cnt) acc.fma(vv[u], xr[u]);
                }
            }
        }
        if (!col_ok) continue;
        if (slot >= 0) {
            acc.store(p.partial + (int64_t)slot * p.d + col);
        } else {
            if (p.agg == CBRS_AGG_MEAN) {
                const int64_t cnt_row = row_e - row_b;
                if (cnt_row > 0) acc.div((float)cnt_row);
            }
            acc.epilogue(p.bias ? p.bias + col : nullptr, p.relu);
            acc.store(p.y + (int64_t)row * p.ldy + col);
            for (int q = 0; q < p.n_peer; ++q) acc.store(p.y_peer[q] + (int64_t)row * p.ldy + col);
        }
    }
}

// heavy rows: add the parked partials in ascending chunk order, then the epilogue
template <int G, int VEC>
__global__ void __launch_bounds__(kSpmmThreads) spmm_heavy_kernel(const SpmmParams p) {
    const int64_t gid = ((int64_t)blockIdx.x * kSpmmThreads + threadIdx.x) / G;
    if (gid >= p.n_heavy) return;
    const int lg = threadIdx.x & (G - 1);
    const int32_t row = p.heavy_row[gid];
    const int64_t s0 = p.heavy_slot_ptr[gid], s1 = p.heavy_slot_ptr[gid + 1];
    for (int c0 = 0; c0 < p.d; c0 += G * VEC) {
        const int col = c0 + lg * VEC;
        if (col >= p.d) continue;
        Vec<VEC> acc;
        acc.zero();
        for (int64_t s = s0; s < s1; ++s) {
            Vec<VEC> t;
            t.load_plain(p.partial + s * p.d + col);
            acc.add(t);
        }
        if (p.agg == CBRS_AGG_MEAN) {
            const int64_t cnt_row = p.rowptr[row + 1] - p.rowptr[row];
            if (cnt_row > 0) acc.div((float)cnt_row);
        }
        acc.epilogue(p.bias ? p.bias + col : nullptr, p.relu);
        acc.store(p.y + (int64_t)row * p.ldy + col);
        for (int q = 0; q < p.n_peer; ++q) acc.store(p.y_peer[q] + (int64_t)row * p.ldy + col);
    }
}

template <int G, int VEC, typename XT = float>
static int launch(const SpmmParams &p, cudaStream_t s) {
    const int64_t threads = p.n_chunks * G;
    if (threads > 0) {
        // row loads in flight per group: 4, or 8 for the half-width bf16 loads of VEC 1 and 4 (the same bytes in
        // flight per lane as the fp32 kernel).  Measured on config 5 (profiles/r01_tune_spmm.log): 4 loads in
        // flight x 32 warps/SM beats 8 x 16 by 1.45x - occupancy, not per-warp MLP, is what saturates HBM here
        constexpr int kLoads = (!std::is_same<XT, float>::value && VEC != 8) ? 8 : 4;
        spmm_chunk_kernel<G, VEC, kLoads, 4, XT><<<(unsigned)cdiv(threads, kSpmmThreads), kSpmmThreads, 0, s>>>(p);
        CBRS_CHECK_LAUNCH("spmm_chunk");
    }
    if (p.n_heavy > 0) {
        spmm_heavy_kernel<G, VEC><<<(unsigned)cdiv(p.n_heavy * G, kSpmmThreads), kSpmmThreads, 0, s>>>(p);
        CBRS_CHECK_LAUNCH("spmm_heavy");
    }
    return CBRS_OK;
}

template <int VEC, typename XT = float>
static int dispatch_g(int lanes_needed, const SpmmParams &p, cudaStream_t s) {
    if (lanes_needed <= 1) return launch<1, VEC, XT>(p, s);
    if (lanes_needed <= 2) return launch<2, VEC, XT>(p, s);
    if (lanes_needed <= 4) return launch<4, VEC, XT>(p, s);
    if (lanes_needed <= 8) return launch<8, VEC, XT>(p, s);
    if (lanes_needed <= 16) return launch<16, VEC, XT>(p, s);
    return launch<32, VEC, XT>(p, s);
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_spmm_workspace_bytes(const cbrs_csr_t *g, int32_t d) {
    if (!g) return 0;
    return align_up((size_t)g->n_slots * (size_t)d * sizeof(float)) + 256;
}

static int spmm_impl(const cbrs_csr_t *g, const void *x, int64_t ldx, void *y, int64_t ldy, int32_t d, int agg,
                     const float *bias, int relu, int dtype, void *const *y_peers_host, int n_peers, void *workspace,
                     size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(g && x && y, CBRS_E_INVALID, "spmm: null argument");
    CBRS_REQUIRE(n_peers >= 0 && n_peers < CBRS_MAX_PEERS && (n_peers == 0 || y_peers_host), CBRS_E_INVALID,
                 "spmm: n_peers=%d (at most %d peer copies)", n_peers, CBRS_MAX_PEERS - 1);
    CBRS_REQUIRE(dtype == CBRS_DTYPE_F32 || dtype == CBRS_DTYPE_BF16, CBRS_E_INVALID, "spmm: dtype=%d", dtype);
    CBRS_REQUIRE(d > 0 && ldx >= d && ldy >= d, CBRS_E_INVALID, "spmm: d=%d ldx=%lld ldy=%lld", d, (long long)ldx,
                 (long long)ldy);
    CBRS_REQUIRE(ldx <= INT32_MAX / 4, CBRS_E_INVALID, "spmm: ldx=%lld (a row stride under 2^31 bytes)", (long long)ldx);
    CBRS_REQUIRE(agg >= CBRS_AGG_WEIGHTED && agg <= CBRS_AGG_MEAN, CBRS_E_INVALID, "spmm: agg=%d", agg);
    CBRS_REQUIRE(g->n_rows >= 0 && g->n_chunks >= 0 && g->chunk_edges > 0, CBRS_E_INVALID, "spmm: bad graph descriptor");
    if (g->n_rows == 0) return CBRS_OK;
    CBRS_REQUIRE(g->rowptr && g->chunk_row && g->chunk_begin && g->chunk_slot && (g->nnz == 0 || g->colidx),
                 CBRS_E_INVALID, "spmm: graph descriptor has null arrays");
    CBRS_REQUIRE(g->n_heavy == 0 || (g->heavy_row && g->heavy_slot_ptr), CBRS_E_INVALID, "spmm: heavy list missing");
    const size_t need = (size_t)g->n_slots * (size_t)d * sizeof(float);
    CBRS_REQUIRE(g->n_slots == 0 || (workspace && workspace_bytes >= need), CBRS_E_WORKSPACE,
                 "spmm: workspace %zu < %zu bytes", workspace_bytes, need);
    SpmmParams p;
    p.rowptr = g->rowptr; p.colidx = g->colidx; p.vals = g->vals;
    p.chunk_row = g->chunk_row; p.chunk_begin = g->chunk_begin; p.chunk_slot = g->chunk_slot; p.chunk_len = g->chunk_len;
    p.n_chunks = g->n_chunks; p.chunk_edges = g->chunk_edges;
    p.x = x; p.ldx = ldx; p.y = (float *)y; p.ldy = ldy; p.d = d; p.agg = agg;
    p.bias = bias; p.relu = relu; p.partial = (float *)workspace;
    p.heavy_row = g->heavy_row; p.heavy_slot_ptr = g->heavy_slot_ptr; p.n_heavy = g->n_heavy;
    bool vec4 = (d % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && ((uintptr_t)x % 16 == 0) &&
                ((uintptr_t)y % 16 == 0) && ((uintptr_t)workspace % 16 == 0) && (!bias || (uintptr_t)bias % 16 == 0);
    p.n_peer = n_peers;
    bool vec4_peers = true;
    for (int q = 0; q < CBRS_MAX_PEERS - 1; ++q) {
        p.y_peer[q] = q < n_peers ? (float *)y_peers_host[q] : nullptr;
        if (q < n_peers) {
            CBRS_REQUIRE(p.y_peer[q], CBRS_E_INVALID, "spmm: peer copy %d is null", q);
            vec4_peers = vec4_peers && ((uintptr_t)p.y_peer[q] % 16 == 0);
        }
    }
    vec4 = vec4 && vec4_peers;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == CBRS_DTYPE_BF16) {
        // a 4-wide bf16 group is an 8-byte load: same lane layout as fp32, half the bytes per edge
        const bool v4 = (d % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && ((uintptr_t)x % 8 == 0) && ((uintptr_t)y % 16 == 0) &&
                        ((uintptr_t)workspace % 16 == 0) && (!bias || (uintptr_t)bias % 16 == 0) && vec4_peers;
        const bool v8 = v4 && (d % 8 == 0) && (ldx % 8 == 0) && ((uintptr_t)x % 16 == 0);
        if (v8) return dispatch_g<8, __nv_bfloat16>(d / 8, p, s);  // 16-byte loads, half the lanes per row
        return v4 ? dispatch_g<4, __nv_bfloat16>(d / 4, p, s) : dispatch_g<1, __nv_bfloat16>(d, p, s);
    }
    return vec4 ? dispatch_g<4>(d / 4, p, s) : dispatch_g<1>(d, p, s);
}

extern "C" int cbrs_spmm_csr(const cbrs_csr_t *g, const void *x, int64_t ldx, void *y, int64_t ldy, int32_t d, int agg,
                             const float *bias, int relu, int dtype, void *workspace, size_t workspace_bytes,
                             void *stream) {
    return spmm_impl(g, x, ldx, y, ldy, d, agg, bias, relu, dtype, nullptr, 0, workspace, workspace_bytes, stream);
}

extern "C" int cbrs_spmm_csr_bcast(const cbrs_csr_t *g, const void *x, int64_t ldx, void *y, int64_t ldy, int32_t d,
                                   int agg, const float *bias, int relu, int dtype, void *const *y_peers_host,
                                   int n_peers, void *workspace, size_t workspace_bytes, void *stream) {
    return spmm_impl(g, x, ldx, y, ldy, d, agg, bias, relu, dtype, y_peers_host, n_peers, workspace, workspace_bytes,
                     stream);
}
