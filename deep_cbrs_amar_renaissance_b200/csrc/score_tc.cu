// bf16 tensor-core catalog scorer + per-user top-k (tcgen05 / TMEM), sm_100a.
//
// Same contract as cbrs_score_catalog_topk (score.cu) - BasicRS classifier with the first
// layer hoisted into P[u] + Q[i] (/root/reference/src/models/basic.py:31-37) - but the
// per-pair GEMM relu(P[u]+Q[i]) @ W2 runs on the 5th-generation tensor cores:
//   * a tile is 128 (user,item) pairs = 4 users x 32 items; thread t produces row t of the
//     A operand, h1 = relu(P[u]+Q[i]) rounded to bf16, straight into shared memory in the
//     canonical K-major SWIZZLE_128B layout (16-byte chunk c of row r at chunk c ^ (r & 7));
//   * W2^T (bf16, K-major, pre-swizzled once by a prep kernel) stays resident in shared memory;
//   * one thread issues ceil(c1/16) tcgen05.mma (M=128, N=c2, K=16) into a TMEM accumulator and
//     commits to an mbarrier;
//   * every thread reads its own accumulator row back with tcgen05.ld (warp w owns TMEM lanes
//     32w..32w+31), applies bias + relu + the output layer + sigmoid and feeds the running
//     per-user top-k lists (same candidate-list scheme as the fp32 kernel).
// There is no warp specialisation inside a CTA: 4+ CTAs are resident per SM (TMEM: 64 of 512
// columns each) and the SM overlaps one CTA's MMA with the others' producer / epilogue phases.
// Precision: h1 and W2 are bf16, accumulation fp32 => scores differ from the fp32 path by
// O(1e-3); the parity tests compare against a bf16-rounding oracle (tolerance stated there).
#include "common.cuh"
#include "tc05.cuh"

#include <string.h>

namespace cbrs {

struct ScoreTcParams {
    const float *P; int64_t ldp;
    const float *Q; int64_t ldq;
    int64_t n_users; int32_t n_items;
    int32_t c1, c2;
    const uint8_t *w2_image;  // [KB][n_pad][128 B] bf16, swizzled
    const float *b2, *w3, *b3;
    int32_t k;
    int32_t *ids_out; float *scores_out;
    const int64_t *excl_rowptr; const int32_t *excl_items;   // exclusion lists (both null: none)
};

constexpr int kTcThreads = 128;
constexpr int kTcTU = 16;  // users per CTA (4 passes of 4 users per item tile)
constexpr int kTcTI = 32;  // items per tile

// W2 [c1, c2] fp32 (Keras [in,out]) -> B operand image: element (n, k) = bf16(W2[k][n]), K-major, SWIZZLE_128B
__global__ void score_tc_prep_kernel(const float *__restrict__ w2, int c1, int c2, int n_pad, int kb_count,
                                     uint8_t *__restrict__ image) {
    const int total = kb_count * n_pad * 64;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int kb = e / (n_pad * 64), rem = e % (n_pad * 64);
        const int n = rem / 64, kk = rem % 64;
        const int kg = kb * 64 + kk;
        const float v = (n < c2 && kg < c1) ? w2[(int64_t)kg * c2 + n] : 0.f;
        const uint32_t off = (uint32_t)kb * n_pad * 128 + tc::sw128_offset(n, kk >> 3) + (kk & 7) * 2;
        *reinterpret_cast<__nv_bfloat16 *>(image + off) = __float2bfloat16_rn(v);
    }
}

// QREG: the classifier's first width fits one 64-wide K block, so a thread keeps its item's Q row
// (64 floats) in registers for all passes of a tile and refills it while the last pass's MMA and
// epilogue are in flight; otherwise Q chunks are re-read (L1) in every pass.
template <bool QREG, bool kExcl>   // kExcl: exclusion lists given
__global__ void __launch_bounds__(kTcThreads, QREG ? 4 : 3) score_tc_kernel(const ScoreTcParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];  // SWIZZLE_128B tiles need 1024-byte alignment
    const int c1 = p.c1;
    const int kb_count = (c1 + 63) / 64;
    const int c1p = kb_count * 64;
    const int n_pad = (p.c2 + 15) / 16 * 16;
    const int cap = topk_list_cap(p.k);
    // carve shared memory (operand tiles first: SWIZZLE_128B needs 1024-byte alignment)
    // (pointers are derived from the __shared__ array without integer round-trips so that the
    //  compiler keeps them in the shared address space: LDS/STS, not generic LD/ST)
    unsigned char *As = smem_raw;                               // [kb][128][128 B]
    unsigned char *Bs = As + kb_count * 16384;                  // [kb][n_pad][128 B]
    float *Ps = reinterpret_cast<float *>(Bs + kb_count * n_pad * 128);  // [TU][c1p]
    float2 *bw = reinterpret_cast<float2 *>(Ps + kTcTU * c1p);  // [n_pad] (b2, w3)
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(bw + n_pad);  // [TU][cap]
    unsigned long long *thr = cand + kTcTU * cap;               // [TU]
    uint64_t *mbar = reinterpret_cast<uint64_t *>(thr + kTcTU);
    int *cnt = reinterpret_cast<int *>(mbar + 1);               // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + kTcTU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t u0 = (int64_t)blockIdx.x * kTcTU;
    const float b3 = __ldg(p.b3);
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < n_pad) tmem_cols <<= 1;

    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 0) {
        tc::mbar_init(mbar, 1);
        tc::fence_mbar_init();
    }
    {   // resident operands
        const int4 *src = reinterpret_cast<const int4 *>(p.w2_image);
        int4 *dst = reinterpret_cast<int4 *>(Bs);
        for (int e = tid; e < kb_count * n_pad * 8; e += kTcThreads) dst[e] = __ldg(src + e);
        for (int e = tid; e < n_pad; e += kTcThreads)
            bw[e] = e < p.c2 ? make_float2(__ldg(p.b2 + e), __ldg(p.w3 + e)) : make_float2(0.f, 0.f);
        for (int e = tid; e < kTcTU * c1p; e += kTcThreads) {
            const int ul = e / c1p, kk = e % c1p;
            Ps[e] = (kk < c1 && u0 + ul < p.n_users) ? __ldg(p.P + (u0 + ul) * p.ldp + kk) : 0.f;
        }
        if (tid < kTcTU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);  // this warp's lane quadrant
    const uint32_t a_addr = tc::smem_u32(As), b_addr = tc::smem_u32(Bs);
    if ((a_addr & 1023u) != 0u) __trap();  // the runtime honours the declared alignment; fail loudly if not
    const uint32_t idesc = tc::idesc_bf16_f32(128, n_pad);
    const int k_steps = (c1 + 15) / 16;       // MMAs per tile (K = 16 each)
    const int chunks = k_steps * 2;           // 16-byte chunks a producer row writes
    uint32_t phase = 0;

    float4 qreg[QREG ? 16 : 1];
    auto load_q = [&](int t0) {
        if (QREG) {
            const int it = t0 + lane;
            const bool ok = it < p.n_items;
            const float *qr = p.Q + (int64_t)(ok ? it : 0) * p.ldq;
#pragma unroll
            for (int j = 0; j < 16; ++j)
                qreg[QREG ? j : 0] = (ok && j * 4 < c1) ? ldg4(qr + j * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    load_q(0);

    for (int t0 = 0; t0 < p.n_items; t0 += kTcTI) {
        for (int ul = warp; ul < kTcTU; ul += kTcThreads / 32)   // user ul is always handled by warp ul % 4
            topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
        const int item = t0 + lane;
        const bool item_ok = item < p.n_items;
        const float *qrow = p.Q + (int64_t)(item_ok ? item : 0) * p.ldq;
        for (int pass = 0; pass < kTcTU / 4; ++pass) {
            const int ul = pass * 4 + warp;
            // ---- producer: row `tid` of the A tile ------------------------------------------
            const float *prow = Ps + ul * c1p;
            if (QREG) {
#pragma unroll
                for (int cg = 0; cg < 8; ++cg) {
                    if (cg < chunks) {
                        const float4 q0 = qreg[QREG ? 2 * cg : 0], q1 = qreg[QREG ? 2 * cg + 1 : 0];
                        const float4 p0 = *reinterpret_cast<const float4 *>(prow + cg * 8);
                        const float4 p1 = *reinterpret_cast<const float4 *>(prow + cg * 8 + 4);
                        uint4 packed;
                        packed.x = tc::pack_bf16x2(fmaxf(p0.x + q0.x, 0.f), fmaxf(p0.y + q0.y, 0.f));
                        packed.y = tc::pack_bf16x2(fmaxf(p0.z + q0.z, 0.f), fmaxf(p0.w + q0.w, 0.f));
                        packed.z = tc::pack_bf16x2(fmaxf(p1.x + q1.x, 0.f), fmaxf(p1.y + q1.y, 0.f));
                        packed.w = tc::pack_bf16x2(fmaxf(p1.z + q1.z, 0.f), fmaxf(p1.w + q1.w, 0.f));
                        if (!item_ok) packed = make_uint4(0u, 0u, 0u, 0u);
                        *reinterpret_cast<uint4 *>(As + tc::sw128_offset(tid, cg)) = packed;
                    }
                }
                if (pass == kTcTU / 4 - 1) load_q(t0 + kTcTI);  // refill under this pass's MMA + epilogue
            } else {
#pragma unroll 2
                for (int cg = 0; cg < chunks; ++cg) {
                    const int kk = cg * 8;
                    uint4 packed = make_uint4(0u, 0u, 0u, 0u);
                    if (kk < c1 && item_ok) {
                        const float4 q0 = ldg4(qrow + kk), q1 = ldg4(qrow + kk + 4);
                        const float4 p0 = *reinterpret_cast<const float4 *>(prow + kk);
                        const float4 p1 = *reinterpret_cast<const float4 *>(prow + kk + 4);
                        packed.x = tc::pack_bf16x2(fmaxf(p0.x + q0.x, 0.f), fmaxf(p0.y + q0.y, 0.f));
                        packed.y = tc::pack_bf16x2(fmaxf(p0.z + q0.z, 0.f), fmaxf(p0.w + q0.w, 0.f));
                        packed.z = tc::pack_bf16x2(fmaxf(p1.x + q1.x, 0.f), fmaxf(p1.y + q1.y, 0.f));
                        packed.w = tc::pack_bf16x2(fmaxf(p1.z + q1.z, 0.f), fmaxf(p1.w + q1.w, 0.f));
                    }
                    *reinterpret_cast<uint4 *>(As + (cg >> 3) * 16384 + tc::sw128_offset(tid, cg & 7)) = packed;
                }
            }
            tc::fence_proxy_async_smem();   // my generic-proxy stores -> visible to the tensor core
            tc::tc_fence_before_sync();     // my previous tcgen05.ld -> ordered before the next MMA
            __syncthreads();
            // ---- MMA: one thread ---------------------------------------------------------------
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after_sync();
                for (int s = 0; s < k_steps; ++s) {
                    const uint32_t koff = (uint32_t)(s & 3) * 32;  // 16 bf16 = 32 bytes inside the swizzle atom
                    const uint64_t da = tc::smem_desc_sw128(a_addr + (s >> 2) * 16384 + koff);
                    const uint64_t db = tc::smem_desc_sw128(b_addr + (s >> 2) * n_pad * 128 + koff);
                    tc::mma_bf16_ss(tmem_base, da, db, idesc, s > 0 ? 1u : 0u);
                }
                tc::mma_commit(mbar);
            }
            tc::mbar_wait(mbar, phase);
            phase ^= 1u;
            tc::tc_fence_after_sync();
            // ---- epilogue: accumulator row `tid` -> logit -> sigmoid -> candidate ----------------
            float logit = 0.f;
            for (int cb = 0; cb < n_pad; cb += 32) {
                uint32_t v0[16], v1[16];
                tc::tmem_ld16(tmem_row + (uint32_t)cb, v0);
                if (cb + 16 < n_pad) tc::tmem_ld16(tmem_row + (uint32_t)cb + 16, v1);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 t = bw[cb + j];
                    logit = fmaf(fmaxf(__uint_as_float(v0[j]) + t.x, 0.f), t.y, logit);
                }
                if (cb + 16 < n_pad) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float2 t = bw[cb + 16 + j];
                        logit = fmaf(fmaxf(__uint_as_float(v1[j]) + t.x, 0.f), t.y, logit);
                    }
                }
            }
            const int64_t user = u0 + ul;
            // candidates are ranked by the logit (sigmoid is monotonic); the sigmoid is applied to the k winners
            if (item_ok && user < p.n_users)
                topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + b3, item, user, p.excl_rowptr, p.excl_items);
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, tmem_cols);
    }
    for (int ul = warp; ul < kTcTU; ul += kTcThreads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

// ---------------------------------------------------------------------------------------------------------
// v2 (first classifier width <= 64, the reference's grids): packed bf16 producer + software pipeline.
//  * P[u] and Q[i] are rounded to bf16 once (Q by the prep kernel into the workspace, P while it is staged in
//    shared memory); a thread keeps its item's Q row as 8 x uint4 (32 registers instead of 64) and builds its A
//    row with add.rn.bf16x2 + max.bf16x2: 8 packed instructions per 16-byte chunk instead of 20 scalar ones.
//    h1 = bf16(bf16(P) + bf16(Q)), relu - the bf16 oracle in the tests does the same roundings;
//  * A tiles and TMEM accumulators are double buffered: the A tile of step s+1 is produced and its MMA issued
//    BEFORE the epilogue of step s, so the tensor core's issue->commit latency hides behind CUDA-core work;
//  * the epilogue reads bias and output-layer weights from shared memory and sums the output layer in eight
//    independent fp32 chains.
struct ScoreTc2Params {
    const float *P; int64_t ldp;
    const uint4 *Qb;            // [n_items_pad][8] : 64 bf16 per item, zero padded
    int64_t n_users; int32_t n_items;
    int32_t c1, c2;
    const uint8_t *w2_image;
    const float *b2, *w3, *b3;
    int32_t k;
    int32_t *ids_out; float *scores_out;
    const int64_t *excl_rowptr; const int32_t *excl_items;   // exclusion lists (both null: none)
};

__global__ void score_tc_qprep_kernel(const float *__restrict__ Q, int64_t ldq, int32_t n_items, int32_t n_items_pad,
                                      int32_t c1, uint4 *__restrict__ Qb) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one 16-byte chunk (8 bf16) per thread
    if (e >= (int64_t)n_items_pad * 8) return;
    const int64_t it = e >> 3;
    const int cg = (int)(e & 7);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int kk = cg * 8 + j;
        v[j] = (it < n_items && kk < c1) ? Q[it * ldq + kk] : 0.f;
    }
    Qb[e] = make_uint4(tc::pack_bf16x2(v[0], v[1]), tc::pack_bf16x2(v[2], v[3]), tc::pack_bf16x2(v[4], v[5]),
                       tc::pack_bf16x2(v[6], v[7]));
}

__device__ __forceinline__ uint32_t bf16x2_add_relu(uint32_t a, uint32_t b) {
    const __nv_bfloat162 x = *reinterpret_cast<const __nv_bfloat162 *>(&a), y = *reinterpret_cast<const __nv_bfloat162 *>(&b);
    const __nv_bfloat162 r = __hmax2(__hadd2(x, y), __float2bfloat162_rn(0.f));
    return *reinterpret_cast<const uint32_t *>(&r);
}

template <bool kExcl>   // exclusion lists given
__global__ void __launch_bounds__(kTcThreads, 4) score_tc2_kernel(const __grid_constant__ ScoreTc2Params p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const int c1 = p.c1;
    const int n_pad = (p.c2 + 15) / 16 * 16;
    const int cap = topk_list_cap(p.k);
    unsigned char *As = smem_raw;                                    // [2][128][128 B]
    unsigned char *Bs = As + 2 * 16384;                              // [n_pad][128 B]
    uint4 *Pb = reinterpret_cast<uint4 *>(Bs + n_pad * 128);         // [TU][8] bf16 rows of P
    float4 *bw = reinterpret_cast<float4 *>(Pb + kTcTU * 8);         // [n_pad/2] (b2[2j], b2[2j+1], w3[2j], w3[2j+1])
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(bw + n_pad / 2);  // [TU][cap]
    unsigned long long *thr = cand + kTcTU * cap;                    // [TU]
    uint64_t *mbar = reinterpret_cast<uint64_t *>(thr + kTcTU);      // [2]
    int *cnt = reinterpret_cast<int *>(mbar + 2);                    // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + kTcTU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t u0 = (int64_t)blockIdx.x * kTcTU;
    const float b3 = __ldg(p.b3);
    uint32_t tmem_cols = 64;
    while ((int)tmem_cols < 2 * n_pad) tmem_cols <<= 1;
    const uint32_t buf_cols = tmem_cols / 2;

    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 0) {
        tc::mbar_init(mbar, 1);
        tc::mbar_init(mbar + 1, 1);
        tc::fence_mbar_init();
    }
    {
        const int4 *src = reinterpret_cast<const int4 *>(p.w2_image);
        int4 *dst = reinterpret_cast<int4 *>(Bs);
        for (int e = tid; e < n_pad * 8; e += kTcThreads) dst[e] = __ldg(src + e);
        for (int e = tid; e < n_pad / 2; e += kTcThreads) {
            const int j0 = 2 * e, j1 = 2 * e + 1;
            bw[e] = make_float4(j0 < p.c2 ? __ldg(p.b2 + j0) : 0.f, j1 < p.c2 ? __ldg(p.b2 + j1) : 0.f,
                                j0 < p.c2 ? __ldg(p.w3 + j0) : 0.f, j1 < p.c2 ? __ldg(p.w3 + j1) : 0.f);
        }
        for (int e = tid; e < kTcTU * 8; e += kTcThreads) {
            const int ul = e >> 3, cg = e & 7;
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int kk = cg * 8 + j;
                v[j] = (kk < c1 && u0 + ul < p.n_users) ? __ldg(p.P + (u0 + ul) * p.ldp + kk) : 0.f;
            }
            Pb[e] = make_uint4(tc::pack_bf16x2(v[0], v[1]), tc::pack_bf16x2(v[2], v[3]), tc::pack_bf16x2(v[4], v[5]),
                               tc::pack_bf16x2(v[6], v[7]));
        }
        if (tid < kTcTU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    const uint32_t a_addr = tc::smem_u32(As), b_addr = tc::smem_u32(Bs);
    if ((a_addr & 1023u) != 0u) __trap();
    const uint32_t idesc = tc::idesc_bf16_f32(128, n_pad);
    const int k_steps = (c1 + 15) / 16;
    const int chunks = k_steps * 2;
    constexpr int kPasses = kTcTU / 4;
    const int n_tiles = (p.n_items + kTcTI - 1) / kTcTI;
    const int n_steps = n_tiles * kPasses;

    uint4 qreg[8];
    auto load_q = [&](int tile) {  // rows are padded to a multiple of 32 items: no bounds check
        const uint4 *qr = p.Qb + ((int64_t)tile * kTcTI + lane) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) qreg[j] = __ldg(qr + j);
    };
    auto produce = [&](int step) {   // A row `tid` of step `step` into buffer step & 1
        const int pass = step % kPasses;
        const uint4 *prow = Pb + (pass * 4 + warp) * 8;
        unsigned char *a = As + (step & 1) * 16384;
#pragma unroll
        for (int cg = 0; cg < 8; ++cg) {
            if (cg < chunks) {
                const uint4 pv = prow[cg];
                const uint4 qv = qreg[cg];
                uint4 h;
                h.x = bf16x2_add_relu(pv.x, qv.x); h.y = bf16x2_add_relu(pv.y, qv.y);
                h.z = bf16x2_add_relu(pv.z, qv.z); h.w = bf16x2_add_relu(pv.w, qv.w);
                *reinterpret_cast<uint4 *>(a + tc::sw128_offset(tid, cg)) = h;
            }
        }
    };
    auto issue = [&](int step) {     // one thread: the MMAs of step `step` into TMEM buffer step & 1
        const uint32_t d = tmem_base + (uint32_t)(step & 1) * buf_cols;
        const uint32_t a = a_addr + (uint32_t)(step & 1) * 16384;
        for (int s = 0; s < k_steps; ++s) {
            const uint32_t koff = (uint32_t)s * 32;
            tc::mma_bf16_ss(d, tc::smem_desc_sw128(a + koff), tc::smem_desc_sw128(b_addr + koff), idesc, s > 0 ? 1u : 0u);
        }
        tc::mma_commit(mbar + (step & 1));
    };

    load_q(0);
    produce(0);
    load_q(kPasses == 1 ? 1 : 0);  // (kPasses > 1: step 1 still belongs to tile 0)
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0 && tc::elect_one()) {   // elected: UTCHMMA issues once, not in a per-lane loop
        tc::tc_fence_after_sync();
        issue(0);
    }
    for (int step = 0; step < n_steps; ++step) {
        const int tile = step / kPasses, pass = step % kPasses;
        const int nxt = step + 1;
        if (pass == 0)
            for (int ul = warp; ul < kTcTU; ul += kTcThreads / 32)
                topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
        if (nxt < n_steps) {
            produce(nxt);                                   // qreg holds the tile of step nxt
            if (nxt % kPasses == kPasses - 1 && nxt + 1 < n_steps) load_q(nxt / kPasses + 1);  // refill for the tile after
        }
        tc::fence_proxy_async_smem();
        tc::tc_fence_before_sync();   // my tcgen05.ld of step-1 precede the MMA that will overwrite that TMEM buffer
        __syncthreads();
        if (warp == 0 && nxt < n_steps && tc::elect_one()) {
            tc::tc_fence_after_sync();
            issue(nxt);
        }
        tc::mbar_wait(mbar + (step & 1), (uint32_t)(step >> 1) & 1u);
        tc::tc_fence_after_sync();
        // ---- epilogue of `step`: accumulator row `tid` ------------------------------------------------------
        const uint32_t trow = tmem_row + (uint32_t)(step & 1) * buf_cols;
        float lacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // independent chains: 4 warps per scheduler hide little latency
        for (int cb = 0; cb < n_pad; cb += 32) {
            uint32_t v0[16], v1[16];
            tc::tmem_ld16(trow + (uint32_t)cb, v0);
            if (cb + 16 < n_pad) tc::tmem_ld16(trow + (uint32_t)cb + 16, v1);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                const float4 t = bw[(cb + j) >> 1];
                lacc[j & 7] = fmaf(fmaxf(__uint_as_float(v0[j]) + t.x, 0.f), t.z, lacc[j & 7]);
                lacc[(j + 1) & 7] = fmaf(fmaxf(__uint_as_float(v0[j + 1]) + t.y, 0.f), t.w, lacc[(j + 1) & 7]);
            }
            if (cb + 16 < n_pad) {
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    const float4 t = bw[(cb + 16 + j) >> 1];
                    lacc[j & 7] = fmaf(fmaxf(__uint_as_float(v1[j]) + t.x, 0.f), t.z, lacc[j & 7]);
                    lacc[(j + 1) & 7] = fmaf(fmaxf(__uint_as_float(v1[j + 1]) + t.y, 0.f), t.w, lacc[(j + 1) & 7]);
                }
            }
        }
        const float logit = ((lacc[0] + lacc[1]) + (lacc[2] + lacc[3])) + ((lacc[4] + lacc[5]) + (lacc[6] + lacc[7]));
        const int ul = pass * 4 + warp;
        const int item = tile * kTcTI + lane;
        const int64_t user = u0 + ul;
        if (item < p.n_items && user < p.n_users)
            topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + b3, item, user, p.excl_rowptr, p.excl_items);
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, tmem_cols);
    }
    for (int ul = warp; ul < kTcTU; ul += kTcThreads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

// ---------------------------------------------------------------------------------------------------------
// v3 (c1 <= 64, c2 <= 64: the reference's grids): every per-pair product on the tensor core, warp-specialised.
// v2 spends ~290 CUDA-core instructions per pair around an 8 kFLOP MMA (0.26 of the bf16 peak): 72 to build the operand
// row in shared memory and 192 for bias + relu + the output dot in fp32.  Here
//  * producers (warps 0-3) form h1 = relu(bf16(P) + bf16(Q)) with one fma.rn.relu.bf16x2 per two elements and write the
//    row straight into TENSOR MEMORY (tcgen05.st; the MMAs read A from there): no operand stores, no swizzle math;
//  * the bias joins the product: the operand has 16 more K columns holding a constant 1 (written once), the image of W2
//    a row holding bf16(b2);
//  * relu + the output layer are a SECOND product: mid warps (4-7) read the accumulator, apply relu, round to bf16
//    (one cvt.rn.relu.bf16x2.f32 per two elements) and store the row as the A operand of an M128 x N16 x K64 MMA
//    against a 16-row image whose row 0 is bf16(w3): the logit arrives in one accumulator column;
//  * final warps (8-11) read that column and feed the per-user candidate lists (same scheme and tie rule as before);
//    warps 12 / 13: one elected thread each issues the MMAs of the first / the output product.  All stages run concurrently on double-buffered TMEM
//    operands / accumulators with mbarriers between them; one CTA per SM (16 users x all items).
// ~125 instructions per pair instead of ~290.  Roundings (the oracle in tests/test_gpu_kernels.py mirrors them):
// h1 = bf16(bf16(P) + bf16(Q)), W2 / b2 / w3 to bf16, h2 = bf16(relu(h1 W2 + b2)) - one more than v2, which kept h2,
// b2 and w3 in fp32; accumulation fp32.
constexpr int kW3Threads = 448;
constexpr int kW3NB = 3;   // pipeline depth: buffers per TMEM operand / accumulator (a step passes 5 stages; with 2 the
                           // loop was latency-bound at ~870 cycles per step, every role waiting half of the time)
// TMEM columns: D1[NB] x 64, D2[NB] x 16, A1[NB] x 32, the shared constant-one K block (8), A2[NB] x 32 = 440 of 512
constexpr uint32_t kW3ColD1 = 0, kW3ColD2 = 192, kW3ColA1 = 240, kW3ColOne = 336, kW3ColA2 = 344;

struct ScoreTc3Params {
    const float *P; int64_t ldp;
    const uint4 *Qb;            // [n_items_pad][8] : 64 bf16 per item, zero padded
    int64_t n_users; int32_t n_items;
    int32_t c1, c2;
    const uint8_t *w_image;     // [2][64][128 B]: bf16(W2^T) K-major SWIZZLE_128B, then the block whose k = 0 column is bf16(b2)
    const uint8_t *w3_image;    // [16][128 B]: row 0 = bf16(w3), rows 1..15 zero
    const float *b3;
    int32_t k;
    int32_t *ids_out; float *scores_out;
    const int64_t *excl_rowptr; const int32_t *excl_items;   // exclusion lists (both null: none)
};

__global__ void score_tc3_prep_kernel(const float *__restrict__ w2, const float *__restrict__ b2, const float *__restrict__ w3,
                                      int c1, int c2, uint8_t *__restrict__ img, uint8_t *__restrict__ img3) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 2 * 64 * 64 + 16 * 64; e += gridDim.x * blockDim.x) {
        if (e < 2 * 64 * 64) {
            const int kb = e >> 12, n = (e >> 6) & 63, kk = e & 63;
            float v = 0.f;
            if (kb == 0) v = (n < c2 && kk < c1) ? w2[(int64_t)kk * c2 + n] : 0.f;
            else v = (kk == 0 && n < c2) ? b2[n] : 0.f;
            *reinterpret_cast<__nv_bfloat16 *>(img + kb * 8192 + tc::sw128_offset(n, kk >> 3) + (kk & 7) * 2) = __float2bfloat16_rn(v);
        } else {
            const int f = e - 2 * 64 * 64, n = f >> 6, kk = f & 63;
            const float v = (n == 0 && kk < c2) ? w3[kk] : 0.f;
            *reinterpret_cast<__nv_bfloat16 *>(img3 + tc::sw128_offset(n, kk >> 3) + (kk & 7) * 2) = __float2bfloat16_rn(v);
        }
    }
}

__device__ __forceinline__ void w3_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void w3_tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
        "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void w3_tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ uint32_t w3_tmem_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void w3_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void w3_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// relu(a * 1 + c) on two bf16 lanes: the exact sum rounded once, then max(., 0) - what add.rn.bf16x2 + max.bf16x2 give
__device__ __forceinline__ uint32_t w3_add_relu(uint32_t a, uint32_t c) {
    uint32_t d;
    asm("fma.rn.relu.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0x3F803F80u), "r"(c));
    return d;
}
// {lo, hi} -> bf16x2 with relu (round to nearest even)
__device__ __forceinline__ uint32_t w3_pack_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

template <bool kExcl>   // exclusion lists given
__global__ void __launch_bounds__(kW3Threads, 1) score_tc3_kernel(const __grid_constant__ ScoreTc3Params p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const int cap = topk_list_cap(p.k);
    unsigned char *W1 = smem_raw;                                    // [2][64][128 B]
    unsigned char *W3 = W1 + 2 * 8192;                               // [16][128 B]
    uint4 *Pb = reinterpret_cast<uint4 *>(W3 + 2048);                // [TU][8] bf16 rows of P
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(Pb + kTcTU * 8);   // [TU][cap]
    unsigned long long *thr = cand + kTcTU * cap;                    // [TU]
    uint64_t *bars = reinterpret_cast<uint64_t *>(thr + kTcTU);      // 8 barriers x NB buffers
    uint64_t *a1_full = bars, *a1_empty = bars + kW3NB, *d1_full = bars + 2 * kW3NB, *d1_empty = bars + 3 * kW3NB;
    uint64_t *a2_full = bars + 4 * kW3NB, *a2_empty = bars + 5 * kW3NB, *d2_full = bars + 6 * kW3NB, *d2_empty = bars + 7 * kW3NB;
    int *cnt = reinterpret_cast<int *>(bars + 8 * kW3NB);            // [TU]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(cnt + kTcTU);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t u0 = (int64_t)blockIdx.x * kTcTU;

    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    if (tid == 32) {
        for (int b = 0; b < kW3NB; ++b) {
            // "full" / "empty" from the CUDA-core side: ONE arrival per warp (lane 0, after __syncwarp) - 32 lanes arriving
            // on the same shared-memory word are 32 serialised atomics per warp, barrier and step
            tc::mbar_init(a1_full + b, 4);  tc::mbar_init(a1_empty + b, 1);
            tc::mbar_init(d1_full + b, 1);  tc::mbar_init(d1_empty + b, 4);
            tc::mbar_init(a2_full + b, 4);  tc::mbar_init(a2_empty + b, 1);
            tc::mbar_init(d2_full + b, 1);  tc::mbar_init(d2_empty + b, 4);
        }
        tc::fence_mbar_init();
    }
    {
        const int4 *src = reinterpret_cast<const int4 *>(p.w_image);
        int4 *dst = reinterpret_cast<int4 *>(W1);
        for (int e = tid; e < 2 * 8192 / 16; e += kW3Threads) dst[e] = __ldg(src + e);
        const int4 *src3 = reinterpret_cast<const int4 *>(p.w3_image);
        int4 *dst3 = reinterpret_cast<int4 *>(W3);
        for (int e = tid; e < 2048 / 16; e += kW3Threads) dst3[e] = __ldg(src3 + e);
        for (int e = tid; e < kTcTU * 8; e += kW3Threads) {
            const int ul = e >> 3, cg = e & 7;
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int kk = cg * 8 + j;
                v[j] = (kk < p.c1 && u0 + ul < p.n_users) ? __ldg(p.P + (u0 + ul) * p.ldp + kk) : 0.f;
            }
            Pb[e] = make_uint4(tc::pack_bf16x2(v[0], v[1]), tc::pack_bf16x2(v[2], v[3]), tc::pack_bf16x2(v[4], v[5]),
                               tc::pack_bf16x2(v[6], v[7]));
        }
        if (tid < kTcTU) { cnt[tid] = 0; thr[tid] = 0ull; }
    }
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    if ((tc::smem_u32(W1) & 1023u) != 0u) __trap();
    constexpr int kPasses = kTcTU / 4;
    const int n_tiles = (p.n_items + kTcTI - 1) / kTcTI;
    const int n_steps = n_tiles * kPasses;
    const uint32_t lane_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);   // this warp's TMEM lane quadrant

    if (warp < 4) {
        // ---------------- producers: thread = pair (user of quadrant `warp`, item `lane`) ----------------
        {   // the constant-one K block every step's product ends with: element 64 = 1, 65..79 = 0 (x the image's bias row)
            const uint32_t one[8] = {0x00003F80u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            w3_tmem_st8(lane_base + kW3ColOne, one);
        }
        uint4 qreg[8], qnext[8];   // this item's Q row, and the next item tile's (requested a whole tile ahead)
        auto load_q = [&](int tile, uint4 (&q)[8]) {   // rows are padded to a multiple of 32 items; past the end: tile 0 again
            const uint4 *qr = p.Qb + ((int64_t)(tile < n_tiles ? tile : 0) * kTcTI + lane) * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) q[j] = __ldg(qr + j);
        };
        load_q(0, qreg);
        int step = 0;
        for (int tile = 0; tile < n_tiles; ++tile) {
            load_q(tile + 1, qnext);
#pragma unroll 1
            for (int pass = 0; pass < kPasses; ++pass, ++step) {
                const int buf = step % kW3NB;
                const uint4 *prow = Pb + (pass * 4 + warp) * 8;
                uint32_t h[32];
#pragma unroll
                for (int cg = 0; cg < 8; ++cg) {
                    const uint4 pv = prow[cg], qv = qreg[cg];
                    h[4 * cg] = w3_add_relu(pv.x, qv.x); h[4 * cg + 1] = w3_add_relu(pv.y, qv.y);
                    h[4 * cg + 2] = w3_add_relu(pv.z, qv.z); h[4 * cg + 3] = w3_add_relu(pv.w, qv.w);
                }
                if (step >= kW3NB) {   // the MMAs that read this operand buffer NB steps ago must have completed
                    tc::mbar_wait(a1_empty + buf, (uint32_t)(step / kW3NB - 1) & 1u);
                    tc::tc_fence_after_sync();
                }
                w3_tmem_st32(lane_base + kW3ColA1 + (uint32_t)buf * 32, h);
                w3_st_wait();
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) w3_arrive(a1_full + buf);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) qreg[j] = qnext[j];
        }
    } else if (warp < 8) {
        // ---------------- mid: accumulator 1 -> relu -> bf16 -> operand of the output product (a second set of mid warps
        // alternating steps measured slower: 53 vs 60 G pairs/s - registers per thread drop to 96) ----------------
        for (int step = 0; step < n_steps; ++step) {
            const int buf = step % kW3NB;
            tc::mbar_wait(d1_full + buf, (uint32_t)(step / kW3NB) & 1u);
            tc::tc_fence_after_sync();
            uint32_t v[64];
#pragma unroll
            for (int cb = 0; cb < 64; cb += 16)
                tc::tmem_ld16(lane_base + kW3ColD1 + (uint32_t)(buf * 64 + cb), *reinterpret_cast<uint32_t(*)[16]>(v + cb));
            tc::tmem_ld_wait();
            tc::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) w3_arrive(d1_empty + buf);
            uint32_t h[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) h[j] = w3_pack_relu(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
            if (step >= kW3NB) {
                tc::mbar_wait(a2_empty + buf, (uint32_t)(step / kW3NB - 1) & 1u);
                tc::tc_fence_after_sync();
            }
            w3_tmem_st32(lane_base + kW3ColA2 + (uint32_t)buf * 32, h);
            w3_st_wait();
            tc::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) w3_arrive(a2_full + buf);
        }
    } else if (warp < 12) {
        // ---------------- final: logit column -> candidate list of the row's user ----------------
        // Exclusion lists (kExcl): a binary search of the user's list per candidate above the threshold (excluded_item).
        // It costs these warps, the pipeline's last stage, +15 % / +21 % kernel time with MovieLens-like / Zipf lists at
        // 4,736 x 200,000 on a B200.  The rival - a bitmask of the tile's listed items, filled by this warp from a per-user
        // cursor before it waits for the logit (no synchronisation with the producer / MMA warps needed) - measured worse:
        // +42 % / +40 %, and +25 % with empty lists, the per-step ballot + reduction on this critical stage costing more
        // than the rare searches (profiles/r03_score_bench_exclusion.jsonl, README there).
        const int quad = warp & 3;
        const float b3 = __ldg(p.b3);
        int step = 0;
        for (int tile = 0; tile < n_tiles; ++tile) {
            for (int ul = quad; ul < kTcTU; ul += 4)   // user ul is only ever touched by the final warp of quadrant ul % 4
                topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
#pragma unroll 1
            for (int pass = 0; pass < kPasses; ++pass, ++step) {
                const int buf = step % kW3NB;
                tc::mbar_wait(d2_full + buf, (uint32_t)(step / kW3NB) & 1u);
                tc::tc_fence_after_sync();
                const float logit = __uint_as_float(w3_tmem_ld1(lane_base + kW3ColD2 + (uint32_t)buf * 16));
                tc::tmem_ld_wait();
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) w3_arrive(d2_empty + buf);
                const int ul = pass * 4 + quad;
                const int item = tile * kTcTI + lane;
                const int64_t user = u0 + ul;
                if (item < p.n_items && user < p.n_users)
                    topk_offer<kExcl>(cand, cnt, thr, cap, ul, logit + b3, item, user, p.excl_rowptr, p.excl_items);
            }
        }
    } else {
        // ---------------- MMA issuers: warp 12 the first product, warp 13 the output product, one elected thread each
        // (one thread for both streams blocks the next step's first product on the previous step's mid stage) ----------------
        if (tc::elect_one()) {
            const uint32_t idesc1 = tc::idesc_bf16_f32(128, 64), idesc2 = tc::idesc_bf16_f32(128, 16);
            const uint32_t w1_addr = tc::smem_u32(W1), w3_addr = tc::smem_u32(W3);
            if (warp == 12) {
                for (int step = 0; step < n_steps; ++step) {
                    const int buf = step % kW3NB;
                    tc::mbar_wait(a1_full + buf, (uint32_t)(step / kW3NB) & 1u);
                    if (step >= kW3NB) tc::mbar_wait(d1_empty + buf, (uint32_t)(step / kW3NB - 1) & 1u);
                    tc::tc_fence_after_sync();
                    const uint32_t d = tmem_base + kW3ColD1 + (uint32_t)buf * 64, a = tmem_base + kW3ColA1 + (uint32_t)buf * 32;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)   // 4 x K=16 of h1 . W2
                        w3_mma_ts(d, a + (uint32_t)ks * 8, tc::smem_desc_sw128(w1_addr + (uint32_t)ks * 32), idesc1, ks > 0 ? 1u : 0u);
                    w3_mma_ts(d, tmem_base + kW3ColOne, tc::smem_desc_sw128(w1_addr + 8192u), idesc1, 1u);   // + 1 . bias row
                    tc::mma_commit(a1_empty + buf);
                    tc::mma_commit(d1_full + buf);
                }
            } else {
                for (int t = 0; t < n_steps; ++t) {
                    const int buf = t % kW3NB;
                    tc::mbar_wait(a2_full + buf, (uint32_t)(t / kW3NB) & 1u);
                    if (t >= kW3NB) tc::mbar_wait(d2_empty + buf, (uint32_t)(t / kW3NB - 1) & 1u);
                    tc::tc_fence_after_sync();
                    const uint32_t d = tmem_base + kW3ColD2 + (uint32_t)buf * 16, a = tmem_base + kW3ColA2 + (uint32_t)buf * 32;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        w3_mma_ts(d, a + (uint32_t)ks * 8, tc::smem_desc_sw128(w3_addr + (uint32_t)ks * 32), idesc2, ks > 0 ? 1u : 0u);
                    tc::mma_commit(a2_empty + buf);
                    tc::mma_commit(d2_full + buf);
                }
            }
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, 512);
    }
    for (int ul = warp; ul < kTcTU; ul += kW3Threads / 32)
        topk_write<true>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

static size_t score_tc3_smem(int k) {
    return 2 * 8192 + 2048 + (size_t)kTcTU * 8 * 16 + topk_lists_smem_bytes(kTcTU, k) + 8 * kW3NB * 8 + 16;
}

static size_t score_tc2_smem(int c2, int k) {
    const int n_pad = (c2 + 15) / 16 * 16;
    return 1024 + 2 * 16384 + (size_t)n_pad * 128 + (size_t)kTcTU * 8 * 16 + (size_t)(n_pad / 2) * 16 +
           topk_lists_smem_bytes(kTcTU, k) + 16 + 16;
}

static size_t score_tc_smem(int c1, int c2, int k) {
    const int kb = (c1 + 63) / 64, n_pad = (c2 + 15) / 16 * 16;
    return 1024 + (size_t)kb * 16384 + (size_t)kb * n_pad * 128 + (size_t)kTcTU * kb * 64 * 4 + (size_t)n_pad * 8 +
           topk_lists_smem_bytes(kTcTU, k) + 8 + 16;
}

}  // namespace cbrs

using namespace cbrs;

static bool score_tc_use_v2(int c1, int c2) { return c1 <= 64 && c2 <= 128; }
static bool score_tc_use_v3(int c1, int c2) { return c1 <= 64 && c2 <= 64; }
constexpr size_t kTc3ImageBytes = 2 * 8192 + 2048;

extern "C" size_t cbrs_score_catalog_topk_bf16_workspace_bytes(int32_t n_items, int32_t c1, int32_t c2) {
    const int kb = (c1 + 63) / 64, n_pad = (c2 + 15) / 16 * 16;
    size_t bytes = align_up((size_t)kb * n_pad * 128);
    if (score_tc_use_v2(c1, c2)) bytes += align_up((size_t)((n_items + kTcTI - 1) / kTcTI) * kTcTI * 128);  // Q as bf16, 128 B per item
    if (c1 <= 64 && c2 <= 64) bytes += align_up(kTc3ImageBytes);   // v3: image of W2 with the bias row, image of w3
    return bytes;
}

extern "C" int cbrs_score_catalog_topk_bf16(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                            int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                            const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                                            float *scores_out, void *workspace, size_t workspace_bytes, void *stream) {
    return cbrs_score_catalog_topk_bf16_ex(P, ldp, Q, ldq, n_users, n_items, c1, w2, b2, c2, w3, b3, k, ids_out, scores_out,
                                           nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cbrs_score_catalog_topk_bf16_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                               int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                               const float *w3, const float *b3, int32_t k, int32_t *ids_out,
                                               float *scores_out, const int64_t *excl_rowptr, const int32_t *excl_items,
                                               void *workspace, size_t workspace_bytes, void *stream) {
    CBRS_REQUIRE(P && Q && w2 && b2 && w3 && b3 && ids_out && scores_out, CBRS_E_INVALID, "score_catalog_bf16: null argument");
    const int rc = check_catalog_args("score_catalog_bf16", excl_rowptr, excl_items, n_users, n_items, k);
    if (rc != CBRS_OK) return rc;
    CBRS_REQUIRE(c1 >= 8 && c1 % 8 == 0 && c1 <= 256 && c2 > 0 && c2 <= 256, CBRS_E_UNSUPPORTED,
                 "score_catalog_bf16: classifier widths c1=%d (multiple of 8, <= 256), c2=%d (<= 256)", c1, c2);
    CBRS_REQUIRE(ldp >= c1 && ldq >= c1 && ldq % 4 == 0 && ((uintptr_t)Q % 16) == 0, CBRS_E_INVALID,
                 "score_catalog_bf16: Q must be 16-byte aligned with ldq %% 4 == 0");
    const size_t need = cbrs_score_catalog_topk_bf16_workspace_bytes(n_items, c1, c2);
    CBRS_REQUIRE(workspace && workspace_bytes >= need && ((uintptr_t)workspace % 16) == 0, CBRS_E_WORKSPACE,
                 "score_catalog_bf16: workspace %zu < %zu bytes", workspace_bytes, need);
    if (n_users == 0) return CBRS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int kb = (c1 + 63) / 64, n_pad = (c2 + 15) / 16 * 16;
    score_tc_prep_kernel<<<32, 256, 0, s>>>(w2, c1, c2, n_pad, kb, (uint8_t *)workspace);
    CBRS_CHECK_LAUNCH("score_tc_prep");
    if (score_tc_use_v2(c1, c2)) {
        const int n_items_pad = (n_items + kTcTI - 1) / kTcTI * kTcTI;
        uint4 *Qb = reinterpret_cast<uint4 *>((uint8_t *)workspace + align_up((size_t)kb * n_pad * 128));
        score_tc_qprep_kernel<<<(unsigned)cdiv((int64_t)n_items_pad * 8, 256), 256, 0, s>>>(Q, ldq, n_items, n_items_pad, c1, Qb);
        CBRS_CHECK_LAUNCH("score_tc_qprep");
        if (score_tc_use_v3(c1, c2)) {
            uint8_t *img = (uint8_t *)workspace + align_up((size_t)kb * n_pad * 128) + align_up((size_t)n_items_pad * 128);
            score_tc3_prep_kernel<<<8, 256, 0, s>>>(w2, b2, w3, c1, c2, img, img + 2 * 8192);
            CBRS_CHECK_LAUNCH("score_tc3_prep");
            ScoreTc3Params p3{P, ldp, Qb, n_users, n_items, c1, c2, img, img + 2 * 8192, b3, k, ids_out, scores_out,
                               excl_rowptr, excl_items};
            return launch_catalog_scorer(score_tc3_kernel<false>, score_tc3_kernel<true>, p3, (unsigned)cdiv(n_users, kTcTU),
                                         kW3Threads, score_tc3_smem(k), 200 * 1024, s, "score_catalog_bf16", "score_tc3");
        }
        ScoreTc2Params p2{P, ldp, Qb, n_users, n_items, c1, c2, (const uint8_t *)workspace, b2, w3, b3, k, ids_out, scores_out,
                          excl_rowptr, excl_items};
        return launch_catalog_scorer(score_tc2_kernel<false>, score_tc2_kernel<true>, p2, (unsigned)cdiv(n_users, kTcTU),
                                     kTcThreads, score_tc2_smem(c2, k), 220 * 1024, s, "score_catalog_bf16", "score_tc2");
    }
    ScoreTcParams p{P, ldp, Q, ldq, n_users, n_items, c1, c2, (const uint8_t *)workspace, b2, w3, b3, k, ids_out, scores_out,
                     excl_rowptr, excl_items};
    const unsigned grid = (unsigned)cdiv(n_users, kTcTU);
    const size_t smem = score_tc_smem(c1, c2, k);
    if (c1 <= 64)
        return launch_catalog_scorer(score_tc_kernel<true, false>, score_tc_kernel<true, true>, p, grid, kTcThreads, smem,
                                     220 * 1024, s, "score_catalog_bf16", "score_tc");
    return launch_catalog_scorer(score_tc_kernel<false, false>, score_tc_kernel<false, true>, p, grid, kTcThreads, smem,
                                 220 * 1024, s, "score_catalog_bf16", "score_tc");
}
