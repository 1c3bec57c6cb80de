// fp32-accurate catalog scorer + per-user top-k on the tensor cores (tcgen05 / TMEM, 3xTF32), sm_100a.
//
// Same contract as cbrs_score_catalog_topk (score.cu) - the BasicRS classifier of /root/reference/src/models/basic.py:31-37
// evaluated for every (user, item) with the first layer hoisted into P[u] + Q[i] - and the same accuracy class: the FFMA
// kernel spends 8.4 kFLOP per pair on the CUDA cores (5.0 G pairs/s = 42 TFLOP/s); here the 64 x 64 product runs on the
// tensor cores WITHOUT giving up fp32 accuracy, by the split the GCN transform uses (dense_tf32.cu):
//      h = relu(P[u] + Q[i]) (fp32)      hh = tf32(h)   hl = h - hh (exact)        W2 = Wh + Wl likewise
//      h W2  ~=  hl Wh + hh Wl + hh Wh         three kind::tf32 MMAs into one fp32 TMEM accumulator
// (the dropped hl Wl term is < 2^-22 |h||w|: scores agree with the fp32 chain to ~1e-6, tests state 1e-5).
//
// A tile is 128 pairs = 4 users x 32 items; the pair (user, item) of TMEM lane 32 q + l is produced by lane l of warps q
// and q + 4 (each takes half of the row's columns) and its Q row stays in their registers for the 4 passes over the
// CTA's 16 users.  The A operand never touches shared memory: a thread writes
// its own row - 64 values of hh, 64 of hl - into TENSOR MEMORY with tcgen05.st (TMEM lane = pair, column = k) and the
// MMAs read A from there (tcgen05.mma [d], [a_tmem], b_desc): no operand stores, no 128-byte swizzle arithmetic, and
// the tensor core's shared-memory reads are the 2 KB W2 slices only (an smem-resident A would cost 4 KB per K = 8 step
// and cap the pipe at 2/3 of its rate).  Wh / Wl sit in shared memory as the K-major SWIZZLE_128B images
// cbrs_dense_tf32x3_prepare writes.  One thread issues the 3 x c1/8 MMAs (M = 128, N = c2, K = 8) and commits to
// mbarriers; an epilogue thread reads its accumulator row back (tcgen05.ld), adds the bias, applies relu and the output
// layer in fp32 and feeds the running per-user top-k lists (the candidate lists of common.cuh, keyed on the logit).
// Operand and accumulator are double buffered in TMEM and the three stages run on their own warps (below).
#include "common.cuh"
#include "tc05.cuh"

#include <stdlib.h>

#include <type_traits>

namespace cbrs {

struct ScoreT3Params {
    const float *P; int64_t ldp;
    const float *Q; int64_t ldq;
    int64_t n_users; int32_t n_items;
    int32_t c1, c2;
    const uint8_t *w_image;   // [2 (hi, lo)][c1/32][c2][128 B] tf32 operand images of W2 (cbrs_dense_tf32x3_prepare)
    const float *b2, *w3, *b3;
    int32_t k;
    int32_t *ids_out; float *scores_out;
    const int64_t *excl_rowptr; const int32_t *excl_items;   // exclusion lists (both null: none)
};

constexpr int kS3TU = 16;   // users per CTA (4 passes of 4 users per item tile)
constexpr int kS3TI = 32;   // items per tile

constexpr int kS3WsThreads = 416;   // warp-specialised kernel: 8 producer warps, the MMA warp, 4 epilogue warps
__device__ __forceinline__ void s3_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// ---------------------------------------------------------------------------------------------------------------------
// Warp-specialised.  The first versions were barrier-synchronous (produce -> __syncthreads -> issue -> mbarrier wait ->
// epilogue, 128 or 256 threads, two CTAs per SM): 15-18 G pairs/s, and ~2,300 cycles per 128-pair step of serialised
// latencies remained with all arithmetic removed (profiles/r02_score_tf32x3_ablation.log); the TMEM budget (A 128 + D 64
// columns per tile) allows only two such CTAs per SM to hide them.  Here ONE CTA per SM (16 users x all items) runs the
// three stages concurrently on double-buffered TMEM operands, with mbarriers between them and no CTA-wide barrier in
// the loop:
//   warps 0-7   producers: warps q and q + 4 own TMEM lane quadrant q (one user of the pass; lane = item) and write half
//               of the row each: h = relu(P[u] + Q[i]) -> tf32 part / remainder -> tcgen05.st into A[step & 1];
//   warp  8     one elected thread issues the 3 x C1/8 MMAs of a step into D[step & 1] and commits twice: A[buf] free,
//               D[buf] full.  (elect.sync, not `lane == 0`: inside a divergent branch ptxas wraps every UTCHMMA in a
//               per-lane loop - ~70 cycles per instruction, which made the issuing thread the bottleneck; elected, the
//               24 MMAs of a step issue in 660 cycles);
//   warps 9-12  epilogue: tcgen05.ld of the row, D[buf] handed back as soon as the loads have returned, then bias, relu,
//               output layer, candidate list of the row's user (user u is only ever touched by warp 9 + u % 4).  (Eight
//               epilogue warps - two per quadrant, partial logits combined through shared memory - measured slower:
//               50.8 vs 47.4 ms at 4736 x 200k.)
template <int C1, int NP, bool kExcl>   // kExcl: exclusion lists given
__global__ void __launch_bounds__(kS3WsThreads, 1) score_tf32x3_ws_kernel(const __grid_constant__ ScoreT3Params p) {
    extern __shared__ __align__(1024) unsigned char s3_smem[];
    constexpr int kAtoms = C1 / 32;
    constexpr int kImage = kAtoms * NP * 128;
    constexpr int E = C1 / 2;                       // operand elements a producer thread writes per row
    constexpr uint32_t kColD = 0, kColA = 2 * NP;   // TMEM: D[2] (NP columns each), then A[2] = (hi C1 | lo C1) each
    constexpr uint32_t kCols = (2 * NP + 4 * C1) <= 128 ? 128u : ((2 * NP + 4 * C1) <= 256 ? 256u : 512u);
    static_assert(2 * NP + 4 * C1 <= 512, "TMEM budget");
    static_assert(E == 16 || E == 32, "a producer thread's slice is one 16- or 32-column TMEM store");
    constexpr int kThreads = kS3WsThreads;
    const int cap = topk_list_cap(p.k);
    unsigned char *Wh = s3_smem;                     // [kAtoms][NP][128 B]
    unsigned char *Wl = Wh + kImage;
    float *Ps = reinterpret_cast<float *>(Wl + kImage);              // [TU][C1]
    float2 *bw = reinterpret_cast<float2 *>(Ps + kS3TU * C1);       // [NP] (b2, w3)
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(bw + NP);   // [TU][cap]
    unsigned long long *thr = cand + kS3TU * cap;                   // [TU]
    uint64_t *bars = reinterpret_cast<uint64_t *>(thr + kS3TU);     // a_full[2], a_empty[2], d_full[2], d_empty[2]
    uint64_t *a_full = bars, *a_empty = bars + 2, *d_full = bars + 4, *d_empty = bars + 6;
    int *cnt = reinterpret_cast<int *>(bars + 8);                   // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + kS3TU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t u0 = (int64_t)blockIdx.x * kS3TU;

    if (warp == 0) tc::tmem_alloc(tmem_slot, kCols);
    if (tid == 32) {
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(a_full + b, 8);      // one arrival per producer warp (lane 0, after the warp's tcgen05.wait::st)
            tc::mbar_init(a_empty + b, 1);     // tcgen05.commit
            tc::mbar_init(d_full + b, 1);      // tcgen05.commit
            tc::mbar_init(d_empty + b, 4);     // one arrival per epilogue warp (32 lanes on one word = 32 serialised atomics)
        }
        tc::fence_mbar_init();
    }
    {   // resident operands
        const int4 *src = reinterpret_cast<const int4 *>(p.w_image);
        int4 *dst = reinterpret_cast<int4 *>(Wh);
        for (int e = tid; e < 2 * kImage / 16; e += kThreads) dst[e] = __ldg(src + e);
        for (int e = tid; e < NP; e += kThreads)
            bw[e] = e < p.c2 ? make_float2(__ldg(p.b2 + e), __ldg(p.w3 + e)) : make_float2(0.f, 0.f);
        for (int e = tid; e < kS3TU * C1; e += kThreads) {
            const int ul = e / C1, kk = e % C1;
            Ps[e] = (u0 + ul < p.n_users) ? __ldg(p.P + (u0 + ul) * p.ldp + kk) : 0.f;
        }
        if (tid < kS3TU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();    // W2 images written through the generic proxy -> visible to the tensor core
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t wh_addr = tc::smem_u32(Wh), wl_addr = tc::smem_u32(Wl);
    if ((wh_addr & 1023u) != 0u) __trap();   // SWIZZLE_128B images need the declared alignment
    constexpr int kPasses = kS3TU / 4;
    const int n_tiles = (p.n_items + kS3TI - 1) / kS3TI;

    if (warp < 8) {
        // ---------------- producers ----------------
        const int quad = warp & 3, kh = warp >> 2;
        const uint32_t trow = tmem_base + ((uint32_t)(quad * 32) << 16) + kColA + (uint32_t)(kh * E);
        float4 qreg[E / 4];   // this thread's half of its item's Q row, kept for the kPasses steps of the item tile
        auto load_q = [&](int tile) {
            const int it = tile * kS3TI + lane;
            const bool ok = it < p.n_items;
            const float *qr = p.Q + (int64_t)(ok ? it : 0) * p.ldq + kh * E;
#pragma unroll
            for (int j = 0; j < E / 4; ++j) qreg[j] = ok ? ldg4(qr + j * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        int step = 0, tile = 0;
        // one step; kLast: the item tile's last pass - the next tile's Q row is requested as soon as this one's last use
        // has been computed, so its latency hides behind the barrier wait and the operand stores
        auto do_pass = [&](int pass, auto last_tag) {
            constexpr bool kLast = decltype(last_tag)::value;
            const int buf = step & 1;
            const float4 *prow = reinterpret_cast<const float4 *>(Ps + (pass * 4 + quad) * C1 + kh * E);
            uint32_t hi[E], lo[E];
#pragma unroll
            for (int j = 0; j < E / 4; ++j) {
                const float4 pv = prow[j], qv = qreg[j];
                const float h0 = fmaxf(pv.x + qv.x, 0.f), h1 = fmaxf(pv.y + qv.y, 0.f);
                const float h2 = fmaxf(pv.z + qv.z, 0.f), h3 = fmaxf(pv.w + qv.w, 0.f);
                const float g0 = tc::tf32_hi(h0), g1 = tc::tf32_hi(h1), g2 = tc::tf32_hi(h2), g3 = tc::tf32_hi(h3);
                hi[4 * j] = __float_as_uint(g0); hi[4 * j + 1] = __float_as_uint(g1);
                hi[4 * j + 2] = __float_as_uint(g2); hi[4 * j + 3] = __float_as_uint(g3);
                lo[4 * j] = __float_as_uint(h0 - g0); lo[4 * j + 1] = __float_as_uint(h1 - g1);
                lo[4 * j + 2] = __float_as_uint(h2 - g2); lo[4 * j + 3] = __float_as_uint(h3 - g3);
            }
            if (kLast) load_q(tile + 1);   // past the catalog: zeros, never used
            if (step >= 2) {   // the MMAs that read this A buffer two steps ago must have completed
                tc::mbar_wait(a_empty + buf, (uint32_t)((step >> 1) - 1) & 1u);
                tc::tc_fence_after_sync();
            }
            const uint32_t ta = trow + (uint32_t)buf * 2 * C1;
            if constexpr (E == 32) {
                tc::tmem_st32(ta, hi);
                tc::tmem_st32(ta + C1, lo);
            } else {
                tc::tmem_st16(ta, hi);
                tc::tmem_st16(ta + C1, lo);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) s3_arrive(a_full + buf);
            ++step;
        };
        load_q(0);
        for (tile = 0; tile < n_tiles; ++tile) {
#pragma unroll 1
            for (int pass = 0; pass < kPasses - 1; ++pass) do_pass(pass, std::false_type{});
            do_pass(kPasses - 1, std::true_type{});
        }
    } else if (warp == 8) {
        // ---------------- MMA issuer: one elected lane (elect.sync: UTCHMMA issued once, no per-lane loop) ----------------
        if (tc::elect_one()) {
            const uint32_t idesc = tc::idesc_tf32_f32(128, NP);
            const int n_steps = n_tiles * kPasses;
            for (int step = 0; step < n_steps; ++step) {
                const int buf = step & 1;
                tc::mbar_wait(a_full + buf, (uint32_t)(step >> 1) & 1u);
                if (step >= 2) tc::mbar_wait(d_empty + buf, (uint32_t)((step >> 1) - 1) & 1u);
                tc::tc_fence_after_sync();
                const uint32_t d = tmem_base + kColD + (uint32_t)buf * NP;
                const uint32_t a = tmem_base + kColA + (uint32_t)buf * 2 * C1;
#pragma unroll
                for (int ks = 0; ks < C1 / 8; ++ks) {   // K = 8 per instruction; small terms first
                    const uint32_t boff = (uint32_t)(ks >> 2) * NP * 128 + (uint32_t)(ks & 3) * 32;
                    const uint64_t dbh = tc::smem_desc_sw128(wh_addr + boff), dbl = tc::smem_desc_sw128(wl_addr + boff);
                    const uint32_t ahi = a + (uint32_t)ks * 8, alo = a + C1 + (uint32_t)ks * 8;
                    tc::mma_tf32_ts(d, alo, dbh, idesc, ks > 0 ? 1u : 0u);
                    tc::mma_tf32_ts(d, ahi, dbl, idesc, 1u);
                    tc::mma_tf32_ts(d, ahi, dbh, idesc, 1u);
                }
                tc::mma_commit(a_empty + buf);   // the operand buffer may be rewritten once these MMAs have read it
                tc::mma_commit(d_full + buf);    // ... and the accumulator is complete
            }
        }
    } else {
        // ---------------- epilogue (warps 9..12: TMEM lane quadrant = warp & 3) ----------------
        // Exclusion lists (kExcl): a binary search of the user's list per candidate above the threshold (excluded_item):
        // +7 % / +10 % kernel time with MovieLens-like / Zipf lists at 4,736 x 200,000 on a B200.  A per-tile bitmask filled
        // by these warps from a per-user cursor measured worse (+12 % / +11 %, +9 % with empty lists;
        // profiles/r03_score_bench_exclusion.jsonl, README there).
        const int quad = warp & 3;
        const float b3 = __ldg(p.b3);
        int step = 0;
        for (int tile = 0; tile < n_tiles; ++tile) {
            // a user's list must have room for the 32 candidates one item tile can add
            for (int ul = quad; ul < kS3TU; ul += 4)   // user ul is only ever touched by warp 9 + ul % 4
                topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
#pragma unroll 1
            for (int pass = 0; pass < kPasses; ++pass, ++step) {
                const int buf = step & 1;
                tc::mbar_wait(d_full + buf, (uint32_t)(step >> 1) & 1u);
                tc::tc_fence_after_sync();
                const uint32_t drow = tmem_base + ((uint32_t)(quad * 32) << 16) + kColD + (uint32_t)(buf * NP);
                uint32_t v[NP];
#pragma unroll
                for (int cb = 0; cb < NP; cb += 16) tc::tmem_ld16(drow + (uint32_t)cb, *reinterpret_cast<uint32_t(*)[16]>(v + cb));
                tc::tmem_ld_wait();
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) s3_arrive(d_empty + buf);      // the accumulator may be overwritten: its values sit in registers
                float lacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // independent chains, fixed combination order
#pragma unroll
                for (int j = 0; j < NP; j += 2) {
                    const float4 t = *reinterpret_cast<const float4 *>(bw + j);   // (b2[j], w3[j], b2[j+1], w3[j+1])
                    lacc[j & 7] = fmaf(fmaxf(__uint_as_float(v[j]) + t.x, 0.f), t.y, lacc[j & 7]);
                    lacc[(j + 1) & 7] = fmaf(fmaxf(__uint_as_float(v[j + 1]) + t.z, 0.f), t.w, lacc[(j + 1) & 7]);
                }
                const float logit = ((lacc[0] + lacc[1]) + (lacc[2] + lacc[3])) + ((lacc[4] + lacc[5]) + (lacc[6] + lacc[7]));
                const int ul = pass * 4 + quad;
                const int item = tile * kS3TI + lane;
                const int64_t user = u0 + ul;
                // candidates are ranked by the logit (sigmoid is monotonic); the sigmoid is applied to the k winners
                if (item < p.n_items && user < p.n_users)
                    topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + b3, item, user, p.excl_rowptr, p.excl_items);
            }
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, kCols);
    }
    for (int ul = warp; ul < kS3TU; ul += kThreads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

static size_t s3_smem_bytes(int c1, int np, int k) {
    return 2 * (size_t)(c1 / 32) * np * 128 + (size_t)kS3TU * c1 * 4 + (size_t)np * 8 + topk_lists_smem_bytes(kS3TU, k) + 8 * 8 + 16;
}

template <int C1, int NP>
static int s3_launch_ws(const ScoreT3Params &p, cudaStream_t s) {
    return launch_catalog_scorer(score_tf32x3_ws_kernel<C1, NP, false>, score_tf32x3_ws_kernel<C1, NP, true>, p,
                                 (unsigned)cdiv(p.n_users, kS3TU), kS3WsThreads, s3_smem_bytes(C1, NP, p.k), 200 * 1024, s,
                                 "score_catalog_tf32x3", "score_catalog_tf32x3");
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_score_catalog_topk_tf32x3_eligible(int32_t c1, int32_t c2) {
    return (c1 == 32 || c1 == 64) && c2 > 0 && c2 <= 64;
}

extern "C" size_t cbrs_score_catalog_topk_tf32x3_workspace_bytes(int32_t c1, int32_t c2) {
    if (!cbrs_score_catalog_topk_tf32x3_eligible(c1, c2)) return 0;
    return 2 * (size_t)(c1 / 32) * ((c2 + 15) / 16 * 16 <= 32 ? 32 : 64) * 128 + (size_t)c1 * 64 * 4;
}

extern "C" int cbrs_score_catalog_topk_tf32x3(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                              int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                              const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                                              void *workspace, size_t workspace_bytes, void *stream) {
    return cbrs_score_catalog_topk_tf32x3_ex(P, ldp, Q, ldq, n_users, n_items, c1, w2, b2, c2, w3, b3, k, ids_out, scores_out,
                                             nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cbrs_score_catalog_topk_tf32x3_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                                 int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                                 const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                                                 float *scores_out, const int64_t *excl_rowptr, const int32_t *excl_items,
                                                 void *workspace, size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(P && Q && w2 && b2 && w3 && b3 && ids_out && scores_out, CBRS_E_INVALID, "score_catalog_tf32x3: null argument");
    const int rc = check_catalog_args("score_catalog_tf32x3", excl_rowptr, excl_items, n_users, n_items, k);
    if (rc != CBRS_OK) return rc;
    CBRS_REQUIRE(cbrs_score_catalog_topk_tf32x3_eligible(c1, c2), CBRS_E_UNSUPPORTED,
                 "score_catalog_tf32x3: classifier widths c1=%d (32 or 64), c2=%d (<= 64); use cbrs_score_catalog_topk", c1, c2);
    CBRS_REQUIRE(ldp >= c1 && ldq >= c1 && ldq % 4 == 0 && ((uintptr_t)Q % 16) == 0, CBRS_E_INVALID,
                 "score_catalog_tf32x3: Q must be 16-byte aligned with ldq %% 4 == 0");
    const size_t need = cbrs_score_catalog_topk_tf32x3_workspace_bytes(c1, c2);
    CBRS_REQUIRE(workspace && workspace_bytes >= need && ((uintptr_t)workspace % 16) == 0, CBRS_E_WORKSPACE,
                 "score_catalog_tf32x3: workspace %zu < %zu bytes", workspace_bytes, need);
    if (n_users == 0) return CBRS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    // W2 [c1, c2] is zero-padded to np columns (a device-to-device strided copy), then split into the two operand images
    const int np = (c2 + 15) / 16 * 16 <= 32 ? 32 : 64;
    uint8_t *image = (uint8_t *)workspace;
    float *w_pad = reinterpret_cast<float *>(image + 2 * (size_t)(c1 / 32) * np * 128);
    const float *w_src = w2;
    if (np != c2) {
        cudaError_t e = cudaMemsetAsync(w_pad, 0, (size_t)c1 * np * 4, s);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(w_pad, (size_t)np * 4, w2, (size_t)c2 * 4, (size_t)c2 * 4, (size_t)c1, cudaMemcpyDeviceToDevice, s);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "score_catalog_tf32x3: padding W2: %s", cudaGetErrorString(e));
        w_src = w_pad;
    }
    const int rc_prep = cbrs_dense_tf32x3_prepare(w_src, c1, np, image, stream);
    if (rc_prep != CBRS_OK) return rc_prep;
    ScoreT3Params p{P, ldp, Q, ldq, n_users, n_items, c1, c2, image, b2, w3, b3, k, ids_out, scores_out, excl_rowptr, excl_items};
    if (c1 == 64) return np == 64 ? s3_launch_ws<64, 64>(p, s) : s3_launch_ws<64, 32>(p, s);
    return np == 64 ? s3_launch_ws<32, 64>(p, s) : s3_launch_ws<32, 32>(p, s);
}
