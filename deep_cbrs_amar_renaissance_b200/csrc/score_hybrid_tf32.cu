// fp32-accurate full-catalog scoring of the FEATURE-BASED hybrid scorer + per-user top-k, chained on the tensor cores
// (tcgen05 / TMEM, 3xTF32), sm_100a.  Same contract as score_hybrid_tc_kernel (score_hybrid_tc.cu): the caller hoists
// the towers and the first layer of dense3a / dense3b into P1 / Q1 / P2 / Q2, and per pair the kernel runs
//      h1 = relu(P1[u] + Q1[i])          h2 = relu(P2[u] + Q2[i])                        (fp32)
//      x1 = relu(h1 W3a2 + b3a2)         x2 = relu(h2 W3b2 + b3b2)
//      g  = relu(x1 Wc1[0:64] + x2 Wc1[64:128] + bc1)
//      logit = relu(g Wc2 + bc2) . wc3 + bc3           -> running per-user top-k, sigmoid on the k winners
// at fp32 accuracy instead of bf16: each of the five 64 x 64 products runs as 3xTF32, as in score_tf32.cu,
//      a W  ~=  al Wh + ah Wl + ah Wh        ah = tf32(a), al = a - ah (exact), W = Wh + Wl likewise
// three kind::tf32 MMAs per K = 8 step into one fp32 TMEM accumulator (the dropped al Wl term is < 2^-22 |a||w|).  Every
// activation that feeds a product (h1, h2, x1, x2, g) is split by the thread that owns its row and written into TENSOR
// memory with tcgen05.st (TMEM lane = pair, column = k; ah in columns 0..63, al in 64..127); the MMAs read A from there.
// Bias, relu, the output dot and the sigmoid stay in fp32 on the CUDA cores.  The weight images are the ones
// cbrs_dense_tf32x3_prepare writes (hi | lo, K-major SWIZZLE_128B), five of them, resident in shared memory.
//
// Organisation, from the resource budget:
//  * Shared memory: the five hi + lo images take 5 x 32 KB = 160 KB, so ONE CTA per SM.  The bf16 chain overlaps one
//    CTA's MMAs with the other CTA's CUDA-core work; here the overlap comes from two warp groups inside the CTA.
//  * Tensor memory: a warp group runs the chain of a 128-pair tile (4 users x 32 items; warp q of the group owns TMEM
//    lane quadrant q = one user, lane l = item l) in 256 columns: A (hi 64 | lo 64), Dx (64), D3 (64), in the order
//      h1 -> Dx -> x1 -> D3 = x1 Wc1a,   h2 -> Dx -> x2 -> D3 += x2 Wc1b,   g -> Dx -> logit
//    i.e. five MMA rounds (24 MMAs each) per tile, each ended by an mbarrier wait.  Two warp groups x 256 columns = all
//    512 columns: the groups score disjoint users (TU / 2 each) over the whole catalog with their own TMEM, mbarrier,
//    named barrier and staged item rows, so they drift apart and one group's MMAs run while the other splits, applies
//    relu and feeds its top-k lists.
//  * Item rows: the 32 items of a tile are the same for the 4 users (warps) of a pass, so their Q1 / Q2 rows are staged
//    in shared memory per warp group (coalesced loads, the next tile's rows in flight in registers), 17 KB per group.
//    Users per CTA TU follows k: candidate lists take TU (2k + 32) x 8 bytes, and at TU = 16 everything fits the 227 KB
//    up to k = 78; above that TU = 8 (1 pass of 4 users per tile and group).  k = 128 runs at TU = 8.
//  * Tensor work: 3 x 40,960 = 122,880 FLOP per pair, which at the data sheet's 1,125 dense TF32 TFLOP/s caps the kernel
//    at about 9 G pairs/s.  Measured on one B200 at 1,000 W (profiles/r04_hybrid_tc_bench.jsonl): 3.74 G pairs/s at
//    6,040 x 3,706 and 4.40 G pairs/s = 540 TFLOP/s at 4,736 x 200,000, 13-17x the generic pair pipeline (0.26 G).
//    Not profiled; the likely bound is the five serialised MMA rounds per tile that only two warp groups hide.
// Top-k: keys (orderable(logit) << 32) | ~item, ties to the lower item id; exclusion lists checked only for a key that
// beats the user's threshold (excluded_item, kExcl).  A pair's arithmetic does not depend on k, on the lists or on the
// other users of its CTA, so results are position invariant and deterministic.
#include "common.cuh"
#include "tc05.cuh"

namespace cbrs {

constexpr int kHfC = 64;                    // width of every hidden layer after the towers
constexpr int kHfThreads = 256;             // two warp groups
constexpr int kHfTI = 32;                   // items per tile
constexpr int kHfImage = 2 * kHfC * kHfC * 4;   // one hi | lo tf32 image of a 64 x 64 weight (cbrs_dense_tf32x3_prepare)
constexpr int kHfQLd = kHfC + 4;            // padded staged Q row: 8 consecutive lanes hit 8 distinct 16-byte bank groups

struct HybridTf32Params {
    const float *P1, *Q1, *P2, *Q2;      // [U, 64], [I, 64], [U, 64], [I, 64] fp32, rows contiguous
    int64_t n_users;
    int32_t n_items;
    const uint8_t *w_images;             // 5 images: W3a2, W3b2, Wc1[0:64], Wc1[64:128], Wc2
    const float *b3a2, *b3b2, *bc1, *bc2, *wc3, *bc3;
    int32_t k;
    int32_t *ids_out;
    float *scores_out;
    const int64_t *excl_rowptr;          // exclusion lists (both null: none)
    const int32_t *excl_items;
};

__device__ __forceinline__ void hf_group_sync(int group) {   // named barrier of one warp group (ids 1, 2)
    asm volatile("bar.sync %0, 128;" ::"r"(group + 1) : "memory");
}

template <int TU, bool kExcl>   // TU: users per CTA (TU / 2 per warp group); kExcl: exclusion lists given
__global__ void __launch_bounds__(kHfThreads, 1) score_hybrid_tf32_kernel(const __grid_constant__ HybridTf32Params p) {
    constexpr int TW = TU / 2;   // users per warp group
    extern __shared__ __align__(1024) unsigned char hf_smem[];
    const int cap = topk_list_cap(p.k);
    unsigned char *Ws = hf_smem;                                          // 5 weight images
    float *P1s = reinterpret_cast<float *>(Ws + 5 * kHfImage);            // [TU][64]
    float *P2s = P1s + TU * kHfC;
    float *bias = P2s + TU * kHfC;                                        // b3a2 | b3b2 | bc1 | bc2 | wc3  (5 x 64)
    float *Qs = bias + 5 * kHfC;                                          // [2 groups][2 tables][TI][kHfQLd]
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(Qs + 4 * kHfTI * kHfQLd);   // [TU][cap]
    unsigned long long *thr = cand + TU * cap;                            // [TU]
    uint64_t *mbar = reinterpret_cast<uint64_t *>(thr + TU);              // [2]: one per warp group
    int *cnt = reinterpret_cast<int *>(mbar + 2);                         // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + TU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int group = warp >> 2, quad = warp & 3, gtid = tid & 127;
    const int64_t cta_u0 = (int64_t)blockIdx.x * TU;
    constexpr uint32_t kCols = 512;   // 2 groups x (A 128 | Dx 64 | D3 64)

    if (warp == 0) tc::tmem_alloc(tmem_slot, kCols);
    if (tid == 32) {
        tc::mbar_init(mbar, 1);
        tc::mbar_init(mbar + 1, 1);
        tc::fence_mbar_init();
    }
    {   // resident operands
        const int4 *src = reinterpret_cast<const int4 *>(p.w_images);
        int4 *dst = reinterpret_cast<int4 *>(Ws);
        for (int e = tid; e < 5 * kHfImage / 16; e += kHfThreads) dst[e] = __ldg(src + e);
        const float *bsrc[5] = {p.b3a2, p.b3b2, p.bc1, p.bc2, p.wc3};
        for (int e = tid; e < 5 * kHfC; e += kHfThreads) bias[e] = __ldg(bsrc[e / kHfC] + e % kHfC);
        for (int e = tid; e < TU * kHfC; e += kHfThreads) {
            const int ul = e / kHfC, kk = e % kHfC;
            const bool ok = cta_u0 + ul < p.n_users;
            P1s[e] = ok ? __ldg(p.P1 + (cta_u0 + ul) * kHfC + kk) : 0.f;
            P2s[e] = ok ? __ldg(p.P2 + (cta_u0 + ul) * kHfC + kk) : 0.f;
        }
        if (tid < TU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();   // weight images written through the generic proxy -> visible to the tensor core
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t ws = tc::smem_u32(Ws);
    if ((ws & 1023u) != 0u) __trap();   // SWIZZLE_128B images need the declared alignment

    // this warp group's TMEM: A hi [0, 64), A lo [64, 128), Dx [128, 192), D3 [192, 256)
    const uint32_t tg = tmem_base + (uint32_t)group * 256u;
    const uint32_t trow = tg + ((uint32_t)(quad * 32) << 16);   // this thread's lane (pair)
    constexpr uint32_t kDx = 128, kD3 = 192;
    const uint32_t idesc = tc::idesc_tf32_f32(128, kHfC);
    uint64_t *bar = mbar + group;
    uint32_t phase = 0;
    const int ub = group * TW;   // this group's first user, CTA-local
    float *Q1s = Qs + group * 2 * kHfTI * kHfQLd, *Q2s = Q1s + kHfTI * kHfQLd;

    // D[d, d + 64) (+)= A W_w, 3xTF32: 8 K-steps of three MMAs, small terms first (as score_tf32.cu)
    auto mma64 = [&](int w, uint32_t d, bool accumulate) {
        const uint32_t wh = ws + (uint32_t)w * kHfImage, wl = wh + kHfImage / 2;
#pragma unroll
        for (int ks = 0; ks < kHfC / 8; ++ks) {
            const uint32_t boff = (uint32_t)(ks >> 2) * kHfC * 128 + (uint32_t)(ks & 3) * 32;
            const uint64_t dbh = tc::smem_desc_sw128(wh + boff), dbl = tc::smem_desc_sw128(wl + boff);
            const uint32_t ahi = tg + (uint32_t)ks * 8, alo = tg + kHfC + (uint32_t)ks * 8;
            tc::mma_tf32_ts(tg + d, alo, dbh, idesc, (accumulate || ks > 0) ? 1u : 0u);
            tc::mma_tf32_ts(tg + d, ahi, dbl, idesc, 1u);
            tc::mma_tf32_ts(tg + d, ahi, dbh, idesc, 1u);
        }
    };
    // the group's A rows are in TMEM: one elected thread issues, everyone waits for completion
    auto round = [&](auto issue) {
        tc::tmem_st_wait();             // my tcgen05.st of the operand have landed
        tc::tc_fence_before_sync();     // ... and my tcgen05.ld of the accumulators are ordered before the next MMA
        hf_group_sync(group);
        if (quad == 0 && tc::elect_one()) {   // elected: UTC*MMA issues once, not in a per-lane loop
            tc::tc_fence_after_sync();
            issue();
            tc::mma_commit(bar);
        }
        tc::mbar_wait(bar, phase);
        phase ^= 1u;
        tc::tc_fence_after_sync();
    };
    // x (64 fp32 values of this thread's row) -> tf32 part into A hi, remainder into A lo
    auto store_split = [&](const float (&x)[kHfC]) {
#pragma unroll
        for (int cb = 0; cb < kHfC; cb += 16) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float h = tc::tf32_hi(x[cb + j]);
                hi[j] = __float_as_uint(h);
                lo[j] = __float_as_uint(x[cb + j] - h);
            }
            tc::tmem_st16(trow + (uint32_t)cb, hi);
            tc::tmem_st16(trow + kHfC + (uint32_t)cb, lo);
        }
    };
    // accumulator columns [col, col + 64) of this thread's row -> relu(d + b)
    auto load_act = [&](uint32_t col, const float *b, float (&x)[kHfC]) {
        uint32_t v[kHfC];
#pragma unroll
        for (int cb = 0; cb < kHfC; cb += 16) tc::tmem_ld16(trow + col + (uint32_t)cb, *reinterpret_cast<uint32_t(*)[16]>(v + cb));
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < kHfC; j += 4) {
            const float4 bb = *reinterpret_cast<const float4 *>(b + j);   // broadcast LDS.128
            x[j] = fmaxf(__uint_as_float(v[j]) + bb.x, 0.f);
            x[j + 1] = fmaxf(__uint_as_float(v[j + 1]) + bb.y, 0.f);
            x[j + 2] = fmaxf(__uint_as_float(v[j + 2]) + bb.z, 0.f);
            x[j + 3] = fmaxf(__uint_as_float(v[j + 3]) + bb.w, 0.f);
        }
    };
    auto add_relu = [](const float *a, const float *b, float (&x)[kHfC]) {
#pragma unroll
        for (int j = 0; j < kHfC; j += 4) {
            const float4 av = *reinterpret_cast<const float4 *>(a + j), bv = *reinterpret_cast<const float4 *>(b + j);
            x[j] = fmaxf(av.x + bv.x, 0.f); x[j + 1] = fmaxf(av.y + bv.y, 0.f);
            x[j + 2] = fmaxf(av.z + bv.z, 0.f); x[j + 3] = fmaxf(av.w + bv.w, 0.f);
        }
    };
    // the tile's Q1 / Q2 rows: 2 tables x 32 items x 16 chunks = 1,024 float4, 8 per thread of the group
    float4 qn[8];
    auto fetch_q = [&](int t0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int f = e * 128 + gtid;
            const int tb = f >> 9, it = (f >> 4) & 31, ch = f & 15;
            const int item = t0 + it;
            const float *src = (tb ? p.Q2 : p.Q1) + (int64_t)(item < p.n_items ? item : 0) * kHfC + ch * 4;
            qn[e] = item < p.n_items ? ldg4(src) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto stage_q = [&]() {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int f = e * 128 + gtid;
            const int tb = f >> 9, it = (f >> 4) & 31, ch = f & 15;
            *reinterpret_cast<float4 *>((tb ? Q2s : Q1s) + it * kHfQLd + ch * 4) = qn[e];
        }
    };
    fetch_q(0);
    const float bc3 = __ldg(p.bc3);

    for (int t0 = 0; t0 < p.n_items; t0 += kHfTI) {
        for (int ul = ub + quad; ul < ub + TW; ul += 4)   // user ul is only ever touched by warp quad of its group
            topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
        const int item = t0 + lane;
        stage_q();          // the group's previous readers of the stage have passed later barriers
        hf_group_sync(group);
        fetch_q(t0 + kHfTI);
        const float *q1 = Q1s + lane * kHfQLd, *q2 = Q2s + lane * kHfQLd;
#pragma unroll 1
        for (int pass = 0; pass < TW / 4; ++pass) {
            const int ul = ub + pass * 4 + quad;
            {
                float x[kHfC];
                add_relu(P1s + ul * kHfC, q1, x);
                store_split(x);
            }
            round([&]() { mma64(0, kDx, false); });          // Dx = h1 W3a2
            {
                float x[kHfC];
                load_act(kDx, bias, x);
                store_split(x);
            }
            round([&]() { mma64(2, kD3, false); });          // D3 = x1 Wc1[0:64]
            {
                float x[kHfC];
                add_relu(P2s + ul * kHfC, q2, x);
                store_split(x);
            }
            round([&]() { mma64(1, kDx, false); });          // Dx = h2 W3b2
            {
                float x[kHfC];
                load_act(kDx, bias + kHfC, x);
                store_split(x);
            }
            round([&]() { mma64(3, kD3, true); });           // D3 += x2 Wc1[64:128]
            {
                float x[kHfC];
                load_act(kD3, bias + 2 * kHfC, x);
                store_split(x);
            }
            round([&]() { mma64(4, kDx, false); });          // Dx = g Wc2
            float logit;
            {
                float x[kHfC];
                load_act(kDx, bias + 3 * kHfC, x);
                float lacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // independent chains, fixed combination order
                const float4 *w3 = reinterpret_cast<const float4 *>(bias + 4 * kHfC);
#pragma unroll
                for (int j = 0; j < kHfC / 4; ++j) {
                    const float4 ww = w3[j];
                    lacc[(4 * j) & 7] = fmaf(x[4 * j], ww.x, lacc[(4 * j) & 7]);
                    lacc[(4 * j + 1) & 7] = fmaf(x[4 * j + 1], ww.y, lacc[(4 * j + 1) & 7]);
                    lacc[(4 * j + 2) & 7] = fmaf(x[4 * j + 2], ww.z, lacc[(4 * j + 2) & 7]);
                    lacc[(4 * j + 3) & 7] = fmaf(x[4 * j + 3], ww.w, lacc[(4 * j + 3) & 7]);
                }
                logit = ((lacc[0] + lacc[1]) + (lacc[2] + lacc[3])) + ((lacc[4] + lacc[5]) + (lacc[6] + lacc[7]));
            }
            const int64_t user = cta_u0 + ul;
            // ranked by the logit (sigmoid is monotonic); the sigmoid is applied to the k winners
            if (item < p.n_items && user < p.n_users)
                topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + bc3, item, user, p.excl_rowptr, p.excl_items);
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, kCols);
    }
    for (int ul = warp; ul < TU; ul += kHfThreads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, cta_u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

static size_t hf_smem_bytes(int k, int tu) {
    return 5 * (size_t)kHfImage + 2 * (size_t)tu * kHfC * 4 + 5 * kHfC * 4 + 4 * (size_t)kHfTI * kHfQLd * 4 +
           topk_lists_smem_bytes(tu, k) + 2 * 8 + 16;
}

template <int TU>
static int hf_launch(const HybridTf32Params &p, cudaStream_t s) {
    return launch_catalog_scorer(score_hybrid_tf32_kernel<TU, false>, score_hybrid_tf32_kernel<TU, true>, p,
                                 (unsigned)cdiv(p.n_users, TU), kHfThreads, hf_smem_bytes(p.k, TU), 227 * 1024, s,
                                 "score_hybrid_topk_tf32x3", "score_hybrid_topk_tf32x3");
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_score_hybrid_topk_tf32x3_workspace_bytes(void) { return 5 * (size_t)kHfImage; }

extern "C" int cbrs_score_hybrid_topk_tf32x3(const float *P1, const float *Q1, const float *P2, const float *Q2,
                                             int64_t n_users, int32_t n_items, int32_t c, const float *w3a2,
                                             const float *b3a2, const float *w3b2, const float *b3b2, const float *wc1,
                                             const float *bc1, const float *wc2, const float *bc2, const float *wc3,
                                             const float *bc3, int32_t k, int32_t *ids_out, float *scores_out,
                                             const int64_t *excl_rowptr, const int32_t *excl_items, void *workspace,
                                             size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(P1 && Q1 && P2 && Q2 && w3a2 && b3a2 && w3b2 && b3b2 && wc1 && bc1 && wc2 && bc2 && wc3 && bc3 && ids_out &&
                     scores_out && workspace,
                 CBRS_E_INVALID, "score_hybrid_topk_tf32x3: null argument");
    const int rc = check_catalog_args("score_hybrid_topk_tf32x3", excl_rowptr, excl_items, n_users, n_items, k);
    if (rc != CBRS_OK) return rc;
    CBRS_REQUIRE(c == kHfC, CBRS_E_UNSUPPORTED, "score_hybrid_topk_tf32x3: built for %d-wide hidden layers (every hybrid grid "
                 "of the reference), got %d", kHfC, c);
    CBRS_REQUIRE(k <= n_items, CBRS_E_INVALID, "score_hybrid_topk_tf32x3: n_users=%lld n_items=%d k=%d", (long long)n_users,
                 n_items, k);
    CBRS_REQUIRE(workspace_bytes >= cbrs_score_hybrid_topk_tf32x3_workspace_bytes() && ((uintptr_t)workspace % 16) == 0,
                 CBRS_E_WORKSPACE, "score_hybrid_topk_tf32x3: workspace too small or misaligned");
    if (n_users == 0) return CBRS_OK;
    uint8_t *image = (uint8_t *)workspace;
    const float *w[5] = {w3a2, w3b2, wc1, wc1 + kHfC * kHfC, wc2};
    for (int m = 0; m < 5; ++m) {
        const int rc_prep = cbrs_dense_tf32x3_prepare(w[m], kHfC, kHfC, image + (size_t)m * kHfImage, stream);
        if (rc_prep != CBRS_OK) return rc_prep;
    }
    HybridTf32Params p;
    p.P1 = P1; p.Q1 = Q1; p.P2 = P2; p.Q2 = Q2; p.n_users = n_users; p.n_items = n_items;
    p.w_images = image;
    p.b3a2 = b3a2; p.b3b2 = b3b2; p.bc1 = bc1; p.bc2 = bc2; p.wc3 = wc3; p.bc3 = bc3;
    p.k = k; p.ids_out = ids_out; p.scores_out = scores_out;
    p.excl_rowptr = excl_rowptr; p.excl_items = excl_items;
    cudaStream_t s = (cudaStream_t)stream;
    // 16 users per CTA while their candidate lists fit beside the images (k <= 78), else 8
    if (hf_smem_bytes(k, 16) <= 227 * 1024) return hf_launch<16>(p, s);
    return hf_launch<8>(p, s);
}
