// Full-catalog scoring of the FEATURE-BASED hybrid scorer + per-user top-k, chained on the tensor cores (tcgen05 / TMEM),
// sm_100a.  Replaces HybridCBRS.call (/root/reference/src/models/hybrid.py:72-89) applied to every (user, item) pair:
//
//   x1 = dense3a([ug || ig])     ug = dense1a(graph emb of u), ig = dense1b(graph emb of i)        (collaborative branch)
//   x2 = dense3b([ub || ib])     ub = dense2a(BERT row of u),  ib = dense2b(BERT row of i)         (content branch)
//   score = sigmoid(clf([x1 || x2]))                dense3a/3b = Dense(c) -> Dense(c), clf = Dense(c) -> Dense(c) -> Dense(1)
//
// Everything that depends on one entity is hoisted by the caller (scoring.py): the four towers and the FIRST layer of
// dense3a / dense3b, whose input is a concatenation of a user part and an item part:
//      h1 = relu(P1[u] + Q1[i]),   h2 = relu(P2[u] + Q2[i])        P* = user half (+ bias), Q* = item half
// Per pair that leaves four c x c products and the output dot - 40 kFLOP at c = 64 - which this kernel runs as a chain
// of tcgen05 MMAs with bf16 operands and fp32 accumulation, the intermediate activations never leaving the SM:
//      D1 = h1 W3a2, D2 = h2 W3b2                      -> x1 = relu(D1 + b), x2 = relu(D2 + b)   (bf16, back to shared memory)
//      D3 = x1 Wc1[0:c] + x2 Wc1[c:2c]                 -> g  = relu(D3 + b)
//      D4 = g Wc2                                      -> logit = relu(D4 + b) . wc3 + bc3 -> running top-k
// A tile is 128 pairs = 4 users x 32 items; thread t owns row t of every operand tile and accumulator (warp w reads
// TMEM lanes 32w..32w+31).  The five weight images stay in shared memory; 256 TMEM columns per CTA, two CTAs per SM, so
// one CTA's MMAs overlap the other's CUDA-core phases (same organisation as score_tc_kernel, score_tc.cu).
// Precision: every operand of an MMA is rounded to bf16 (nearest even), sums are fp32; the parity test compares against
// an oracle that rounds at the same points (tests/test_gpu_hybrid_catalog.py, tolerance stated there).  Top-k: exact on
// the kernel's own scores, ties to the lower item id (the candidate lists of common.cuh).
#include "common.cuh"
#include "tc05.cuh"

namespace cbrs {

constexpr int kHyC = 64;         // width of every hidden layer after the towers (all hybrid grids of the reference)
constexpr int kHyThreads = 128;
// users per CTA = template parameter TU (TU / 4 passes of 4 users per item tile): 16, or 24 / 32 when that brings the
// grid down to one wave of 2 CTAs per SM (6,040 users: 378 CTAs on 296 slots with 16, 252 with 24)
constexpr int kHyTI = 32;        // items per tile
constexpr int kHyTile = 128 * 128;   // one 128-row x 64-bf16 operand tile
constexpr int kHyW = kHyC * 128;     // one 64 x 64 bf16 weight image

struct HybridTcParams {
    const float *P1, *Q1, *P2, *Q2;      // [U, 64], [I, 64], [U, 64], [I, 64] fp32, rows contiguous (ld = 64)
    int64_t n_users;
    int32_t n_items;
    const uint8_t *w_images;             // 5 x [64][128 B] bf16, SWIZZLE_128B: W3a2, W3b2, Wc1a, Wc1b, Wc2
    const float *b3a2, *b3b2, *bc1, *bc2, *wc3, *bc3;
    int32_t k;
    int32_t *ids_out;
    float *scores_out;
    const int64_t *excl_rowptr;          // exclusion lists (both null: none)
    const int32_t *excl_items;
};

// W [64 (in), 64 (out)] fp32, Keras layout, row stride ldw -> B operand image: element (n, kk) = bf16(W[kk][n])
__global__ void hy_prep_kernel(const float *w3a2, const float *w3b2, const float *wc1, const float *wc2, uint8_t *image) {
    const float *src[5] = {w3a2, w3b2, wc1, wc1 + kHyC * kHyC, wc2};
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 5 * kHyC * kHyC; e += gridDim.x * blockDim.x) {
        const int m = e / (kHyC * kHyC), rem = e % (kHyC * kHyC);
        const int kk = rem / kHyC, n = rem % kHyC;
        const uint32_t off = (uint32_t)m * kHyW + tc::sw128_offset(n, kk >> 3) + (kk & 7) * 2;
        *reinterpret_cast<__nv_bfloat16 *>(image + off) = __float2bfloat16_rn(src[m][kk * kHyC + n]);
    }
}

// row `tid` of an A tile: f(cg, v) fills the 8 (already activated) fp32 values of 16-byte chunk cg; rounded to bf16
template <typename F>
__device__ __forceinline__ void hy_store_row(unsigned char *tile, int tid, bool live, F f) {
#pragma unroll
    for (int cg = 0; cg < 8; ++cg) {
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
        if (live) {
            float v[8];
            f(cg, v);
            packed.x = tc::pack_bf16x2(v[0], v[1]);
            packed.y = tc::pack_bf16x2(v[2], v[3]);
            packed.z = tc::pack_bf16x2(v[4], v[5]);
            packed.w = tc::pack_bf16x2(v[6], v[7]);
        }
        *reinterpret_cast<uint4 *>(tile + tc::sw128_offset(tid, cg)) = packed;
    }
}

constexpr int kHyQLd = kHyC + 4;   // padded row of the staged Q tile: 8 consecutive lanes hit 8 distinct 16-byte bank groups

template <int TU, bool kExcl>   // kExcl: exclusion lists given
__global__ void __launch_bounds__(kHyThreads, 2) score_hybrid_tc_kernel(const HybridTcParams p) {
    extern __shared__ __align__(1024) unsigned char hy_smem[];
    const int cap = topk_list_cap(p.k);
    unsigned char *A1 = hy_smem;                               // [128][128 B]
    unsigned char *A2 = A1 + kHyTile;
    unsigned char *Ws = A2 + kHyTile;                          // 5 weight images
    float *P1s = reinterpret_cast<float *>(Ws + 5 * kHyW);     // [TU][64]
    float *P2s = P1s + TU * kHyC;
    float *bias = P2s + TU * kHyC;                          // b3a2 | b3b2 | bc1 | bc2 | wc3  (5 x 64)
    float *Q1s = bias + 5 * kHyC;                              // [TI][kHyQLd]: the tile's item halves, shared by all 4 users
    float *Q2s = Q1s + kHyTI * kHyQLd;
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(Q2s + kHyTI * kHyQLd);   // [TU][cap]
    unsigned long long *thr = cand + TU * cap;              // [TU]
    uint64_t *mbar = reinterpret_cast<uint64_t *>(thr + TU);
    int *cnt = reinterpret_cast<int *>(mbar + 1);              // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + TU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t u0 = (int64_t)blockIdx.x * TU;
    const float bc3 = __ldg(p.bc3);
    constexpr uint32_t kCols = 256;   // D1 | D2 | D3 | D4, 64 fp32 columns each

    if (warp == 0) tc::tmem_alloc(tmem_slot, kCols);
    if (tid == 0) {
        tc::mbar_init(mbar, 1);
        tc::fence_mbar_init();
    }
    {   // resident operands
        const int4 *src = reinterpret_cast<const int4 *>(p.w_images);
        int4 *dst = reinterpret_cast<int4 *>(Ws);
        for (int e = tid; e < 5 * kHyW / 16; e += kHyThreads) dst[e] = __ldg(src + e);
        const float *bsrc[5] = {p.b3a2, p.b3b2, p.bc1, p.bc2, p.wc3};
        for (int e = tid; e < 5 * kHyC; e += kHyThreads) bias[e] = __ldg(bsrc[e / kHyC] + e % kHyC);
        for (int e = tid; e < TU * kHyC; e += kHyThreads) {
            const int ul = e / kHyC, kk = e % kHyC;
            const bool ok = u0 + ul < p.n_users;
            P1s[e] = ok ? __ldg(p.P1 + (u0 + ul) * kHyC + kk) : 0.f;
            P2s[e] = ok ? __ldg(p.P2 + (u0 + ul) * kHyC + kk) : 0.f;
        }
        if (tid < TU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    const uint32_t a1 = tc::smem_u32(A1), a2 = tc::smem_u32(A2), ws = tc::smem_u32(Ws);
    if ((a1 & 1023u) != 0u) __trap();
    const uint32_t idesc = tc::idesc_bf16_f32(128, kHyC);
    uint32_t phase = 0;

    // one product A[128 x 64] . W[64 x 64] into TMEM columns [col, col + 64): 4 MMAs of K = 16
    auto mma64 = [&](uint32_t a_addr, int w_index, uint32_t col, bool accumulate) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const uint32_t koff = (uint32_t)s * 32;
            tc::mma_bf16_ss(tmem_base + col, tc::smem_desc_sw128(a_addr + koff),
                            tc::smem_desc_sw128(ws + (uint32_t)w_index * kHyW + koff), idesc, (accumulate || s > 0) ? 1u : 0u);
        }
    };
    // hand the operand tiles to the tensor core, run `issue` on one thread, wait for completion
    auto round = [&](auto issue) {
        tc::fence_proxy_async_smem();   // my generic-proxy stores -> visible to the tensor core
        tc::tc_fence_before_sync();     // my previous tcgen05.ld -> ordered before the next MMA
        __syncthreads();
        if (warp == 0 && tc::elect_one()) {   // elected: UTCHMMA issues once, not in a per-lane loop
            tc::tc_fence_after_sync();
            issue();
            tc::mma_commit(mbar);
        }
        tc::mbar_wait(mbar, phase);
        phase ^= 1u;
        tc::tc_fence_after_sync();
    };
    // accumulator columns [col, col + 64) of row tid -> relu(d + b) as 64 floats in registers
    auto load_act = [&](uint32_t col, const float *b, float (&x)[kHyC]) {
#pragma unroll
        for (int cb = 0; cb < kHyC; cb += 16) {
            uint32_t v[16];
            tc::tmem_ld16(tmem_row + col + (uint32_t)cb, v);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
                const float4 bb = *reinterpret_cast<const float4 *>(b + cb + j);   // broadcast LDS.128
                x[cb + j] = fmaxf(__uint_as_float(v[j]) + bb.x, 0.f);
                x[cb + j + 1] = fmaxf(__uint_as_float(v[j + 1]) + bb.y, 0.f);
                x[cb + j + 2] = fmaxf(__uint_as_float(v[j + 2]) + bb.z, 0.f);
                x[cb + j + 3] = fmaxf(__uint_as_float(v[j + 3]) + bb.w, 0.f);
            }
        }
    };
    // The 32 items of a tile are the same for all 4 users (warps): their Q1 / Q2 rows are staged in shared memory once
    // per tile (coalesced 128-bit loads, 8 per thread) instead of 128 scalar L1 loads per thread and pass.  The next
    // tile's rows travel in registers while the current tile is computed.
    float4 qn[8];
    auto fetch_q = [&](int t0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int f = e * kHyThreads + tid;          // 0 .. 1023: table (512 float4 each), item, chunk
            const int tb = f >> 9, it = (f >> 4) & 31, ch = f & 15;
            const int item = t0 + it;
            const float *src = (tb ? p.Q2 : p.Q1) + (int64_t)(item < p.n_items ? item : 0) * kHyC + ch * 4;
            qn[e] = item < p.n_items ? ldg4(src) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto stage_q = [&]() {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int f = e * kHyThreads + tid;
            const int tb = f >> 9, it = (f >> 4) & 31, ch = f & 15;
            *reinterpret_cast<float4 *>((tb ? Q2s : Q1s) + it * kHyQLd + ch * 4) = qn[e];
        }
    };
    fetch_q(0);

    for (int t0 = 0; t0 < p.n_items; t0 += kHyTI) {
        for (int ul = warp; ul < TU; ul += kHyThreads / 32)   // user ul is always handled by warp ul % 4
            topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
        const int item = t0 + lane;
        const bool item_ok = item < p.n_items;
        stage_q();                 // every warp is past the previous tile's producer phases (it passed later barriers)
        __syncthreads();
        fetch_q(t0 + kHyTI);       // next tile's rows: in flight during this tile's 4 passes
        const float *q1 = Q1s + lane * kHyQLd, *q2 = Q2s + lane * kHyQLd;
        for (int pass = 0; pass < TU / 4; ++pass) {
            const int ul = pass * 4 + warp;
            const float *p1 = P1s + ul * kHyC, *p2 = P2s + ul * kHyC;
            // ---- h1, h2: first layers of dense3a / dense3b (hoisted halves added here) ----
            auto add_relu = [](const float *a, const float *b, int cg, float (&v)[8]) {
                const float4 a0 = *reinterpret_cast<const float4 *>(a + cg * 8), a1v = *reinterpret_cast<const float4 *>(a + cg * 8 + 4);
                const float4 b0 = *reinterpret_cast<const float4 *>(b + cg * 8), b1v = *reinterpret_cast<const float4 *>(b + cg * 8 + 4);
                v[0] = fmaxf(a0.x + b0.x, 0.f); v[1] = fmaxf(a0.y + b0.y, 0.f); v[2] = fmaxf(a0.z + b0.z, 0.f); v[3] = fmaxf(a0.w + b0.w, 0.f);
                v[4] = fmaxf(a1v.x + b1v.x, 0.f); v[5] = fmaxf(a1v.y + b1v.y, 0.f); v[6] = fmaxf(a1v.z + b1v.z, 0.f); v[7] = fmaxf(a1v.w + b1v.w, 0.f);
            };
            hy_store_row(A1, tid, item_ok, [&](int cg, float (&v)[8]) { add_relu(p1, q1, cg, v); });
            hy_store_row(A2, tid, item_ok, [&](int cg, float (&v)[8]) { add_relu(p2, q2, cg, v); });
            round([&]() {
                mma64(a1, 0, 0, false);      // D1 = h1 W3a2
                mma64(a2, 1, 64, false);     // D2 = h2 W3b2
            });
            {   // x1, x2 -> operand tiles (the MMAs that read h1 / h2 have completed)
                float x[kHyC];
                load_act(0, bias, x);
                hy_store_row(A1, tid, true, [&](int cg, float (&v)[8]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = x[cg * 8 + j];
                });
                load_act(64, bias + kHyC, x);
                hy_store_row(A2, tid, true, [&](int cg, float (&v)[8]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = x[cg * 8 + j];
                });
            }
            round([&]() {
                mma64(a1, 2, 128, false);    // D3 = x1 Wc1[0:c]
                mma64(a2, 3, 128, true);     //    + x2 Wc1[c:2c]
            });
            {
                float x[kHyC];
                load_act(128, bias + 2 * kHyC, x);
                hy_store_row(A1, tid, true, [&](int cg, float (&v)[8]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = x[cg * 8 + j];
                });
            }
            round([&]() { mma64(a1, 4, 192, false); });   // D4 = g Wc2
            float logit = 0.f;
            {
                float x[kHyC];
                load_act(192, bias + 3 * kHyC, x);
                const float4 *w3 = reinterpret_cast<const float4 *>(bias + 4 * kHyC);
#pragma unroll
                for (int j = 0; j < kHyC / 4; ++j) {
                    const float4 ww = w3[j];
                    logit = fmaf(x[4 * j], ww.x, logit);
                    logit = fmaf(x[4 * j + 1], ww.y, logit);
                    logit = fmaf(x[4 * j + 2], ww.z, logit);
                    logit = fmaf(x[4 * j + 3], ww.w, logit);
                }
            }
            const int64_t user = u0 + ul;
            // ranked by the logit (sigmoid is monotonic); the sigmoid is applied to the k winners
            if (item_ok && user < p.n_users)
                topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + bc3, item, user, p.excl_rowptr, p.excl_items);
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, kCols);
    }
    for (int ul = warp; ul < TU; ul += kHyThreads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

static size_t hy_smem_bytes(int k, int tu) {
    return 2 * (size_t)kHyTile + 5 * (size_t)kHyW + 2 * tu * kHyC * 4 + 5 * kHyC * 4 + 2 * (size_t)kHyTI * kHyQLd * 4 +
           topk_lists_smem_bytes(tu, k) + 8 + 16;
}

template <int TU>
static int hy_launch(const HybridTcParams &p, cudaStream_t s) {
    return launch_catalog_scorer(score_hybrid_tc_kernel<TU, false>, score_hybrid_tc_kernel<TU, true>, p,
                                 (unsigned)cdiv(p.n_users, TU), kHyThreads, hy_smem_bytes(p.k, TU), 227 * 1024, s,
                                 "score_hybrid_topk_bf16", "score_hybrid_topk_bf16");
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_score_hybrid_topk_bf16_workspace_bytes(void) { return 5 * (size_t)kHyW + 256; }

extern "C" int cbrs_score_hybrid_topk_bf16(const float *P1, const float *Q1, const float *P2, const float *Q2, int64_t n_users,
                                           int32_t n_items, int32_t c, const float *w3a2, const float *b3a2, const float *w3b2,
                                           const float *b3b2, const float *wc1, const float *bc1, const float *wc2,
                                           const float *bc2, const float *wc3, const float *bc3, int32_t k, int32_t *ids_out,
                                           float *scores_out, void *workspace, size_t workspace_bytes, void *stream) {
    return cbrs_score_hybrid_topk_bf16_ex(P1, Q1, P2, Q2, n_users, n_items, c, w3a2, b3a2, w3b2, b3b2, wc1, bc1, wc2, bc2, wc3,
                                          bc3, k, ids_out, scores_out, nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cbrs_score_hybrid_topk_bf16_ex(const float *P1, const float *Q1, const float *P2, const float *Q2,
                                              int64_t n_users, int32_t n_items, int32_t c, const float *w3a2,
                                              const float *b3a2, const float *w3b2, const float *b3b2, const float *wc1,
                                              const float *bc1, const float *wc2, const float *bc2, const float *wc3,
                                              const float *bc3, int32_t k, int32_t *ids_out, float *scores_out,
                                              const int64_t *excl_rowptr, const int32_t *excl_items, void *workspace,
                                              size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(P1 && Q1 && P2 && Q2 && w3a2 && b3a2 && w3b2 && b3b2 && wc1 && bc1 && wc2 && bc2 && wc3 && bc3 && ids_out &&
                     scores_out && workspace,
                 CBRS_E_INVALID, "score_hybrid_topk_bf16: null argument");
    const int rc = check_catalog_args("score_hybrid_topk_bf16", excl_rowptr, excl_items, n_users, n_items, k);
    if (rc != CBRS_OK) return rc;
    CBRS_REQUIRE(c == kHyC, CBRS_E_UNSUPPORTED, "score_hybrid_topk_bf16: built for %d-wide hidden layers (every hybrid grid of the "
                 "reference), got %d", kHyC, c);
    CBRS_REQUIRE(k <= n_items, CBRS_E_INVALID, "score_hybrid_topk_bf16: n_users=%lld n_items=%d k=%d", (long long)n_users,
                 n_items, k);
    CBRS_REQUIRE(workspace_bytes >= cbrs_score_hybrid_topk_bf16_workspace_bytes() && ((uintptr_t)workspace % 16) == 0,
                 CBRS_E_WORKSPACE, "score_hybrid_topk_bf16: workspace too small or misaligned");
    if (n_users == 0) return CBRS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    hy_prep_kernel<<<20, 256, 0, s>>>(w3a2, w3b2, wc1, wc2, (uint8_t *)workspace);
    CBRS_CHECK_LAUNCH("score_hybrid_prep");
    HybridTcParams p;
    p.P1 = P1; p.Q1 = Q1; p.P2 = P2; p.Q2 = Q2; p.n_users = n_users; p.n_items = n_items;
    p.w_images = (const uint8_t *)workspace;
    p.b3a2 = b3a2; p.b3b2 = b3b2; p.bc1 = bc1; p.bc2 = bc2; p.wc3 = wc3; p.bc3 = bc3;
    p.k = k; p.ids_out = ids_out; p.scores_out = scores_out;
    p.excl_rowptr = excl_rowptr; p.excl_items = excl_items;
    // users per CTA: 16, unless 24 or 32 bring the grid down to one wave (2 CTAs per SM) - a second, part-filled wave
    // costs as much as a full one
    const int64_t slots = 2 * kSMs;
    const size_t two_per_sm = (228 * 1024 - 2 * 1024) / 2;   // two CTAs (+ 1 KB reserved each) in an SM's 228 KB
    if (cdiv(n_users, 16) > slots && cdiv(n_users, 24) <= slots && hy_smem_bytes(k, 24) <= two_per_sm) return hy_launch<24>(p, s);
    if (cdiv(n_users, 16) > slots && cdiv(n_users, 32) <= slots && hy_smem_bytes(k, 32) <= two_per_sm) return hy_launch<32>(p, s);
    return hy_launch<16>(p, s);
}
