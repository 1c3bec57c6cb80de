// Fused full-catalog scorer + per-user top-k for the BasicRS classifier (fp32).  Row T (catalog
// form) with rows S1/S2 folded in.
//
// The reference never scores the whole catalog (it ranks the test pairs only,
// /root/reference/src/experiment.py:197-207); parity is "reference scorer
// (src/models/basic.py:31-37) on every (user, item) + stable descending sort".
//
// Everything that depends on one entity is hoisted by the caller with cbrs_dense:
//   P[u,:] = unet(emb[u]) @ W1[:du] + b1      Q[i,:] = inet(emb[i]) @ W1[du:]
// so that the classifier's first layer on [u' || i'] is relu(P[u] + Q[i]).  Per pair the kernel
// computes h2 = relu(relu(P[u]+Q[i]) @ W2 + b2), logit = h2.w3 + b3, sigmoid, and keeps a running
// top-k per user in shared memory - the U x I score matrix is never written.
//
// CTA = 16 users; the item catalog streams through shared memory in tiles of 32 items
// (transposed, 128-bit reads).  Each thread owns 1 user x 8 items x 8 classifier columns:
// 64 FFMA per 3 LDS.128 + 16 add/max.  Candidates above the user's current k-th score go to
// the per-user candidate lists of common.cuh, keyed on the sigmoid score.
#include "common.cuh"

namespace cbrs {

struct ScoreParams {
    const float *P; int64_t ldp;
    const float *Q; int64_t ldq;
    int64_t n_users; int32_t n_items;
    int32_t c1, c2;
    const float *w2, *b2, *w3, *b3;
    int32_t k;
    int32_t *ids_out; float *scores_out;
    const int64_t *excl_rowptr; const int32_t *excl_items;   // exclusion lists (both null: none)
};

constexpr int kScThreads = 256;
constexpr int kScTU = 16;       // users per CTA
constexpr int kScTI = 32;       // items per tile
constexpr int kScQS = kScTI + 4;  // padded row of the transposed item tile

// CT: threads across the classifier's second-layer columns: 8 (c2 <= 64) or 16 (c2 <= 128); kExcl: exclusion lists given
template <int CT, bool kExcl>
__global__ void __launch_bounds__(kScThreads, 2) score_catalog_kernel(const ScoreParams p) {
    constexpr int PG = kScThreads / CT;  // pair groups (1 user x 8 items each)
    constexpr int UPP = PG / 4;          // users per pass (a user's 32 items = 4 groups)
    constexpr int C2P = CT * 8;          // padded second-layer width
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int c1 = p.c1;
    const int cap = topk_list_cap(p.k);
    float *Ws = reinterpret_cast<float *>(smem_raw);       // [c1][C2P]
    float *Ps = Ws + c1 * C2P;                              // [kScTU][c1]
    float *Qs = Ps + kScTU * c1;                            // [c1][kScQS] (transposed tile)
    float *b2s = Qs + c1 * kScQS;                           // [C2P]
    float *w3s = b2s + C2P;                                 // [C2P]
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(w3s + C2P);  // [kScTU][cap]
    unsigned long long *thr = cand + kScTU * cap;           // [kScTU]
    int *cnt = reinterpret_cast<int *>(thr + kScTU);        // [kScTU]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ct = tid % CT, pg = tid / CT;
    const int user_in_pass = pg >> 2, item_oct = pg & 3;
    const int64_t u0 = (int64_t)blockIdx.x * kScTU;
    const float b3 = __ldg(p.b3);

    for (int e = tid; e < c1 * C2P; e += kScThreads) {
        const int kk = e / C2P, n = e % C2P;
        Ws[e] = n < p.c2 ? __ldg(p.w2 + (int64_t)kk * p.c2 + n) : 0.f;
    }
    for (int e = tid; e < C2P; e += kScThreads) {
        b2s[e] = e < p.c2 ? __ldg(p.b2 + e) : 0.f;
        w3s[e] = e < p.c2 ? __ldg(p.w3 + e) : 0.f;
    }
    for (int e = tid; e < kScTU * c1; e += kScThreads) {
        const int ul = e / c1, kk = e % c1;
        Ps[e] = (u0 + ul < p.n_users) ? __ldg(p.P + (u0 + ul) * p.ldp + kk) : 0.f;
    }
    if (tid < kScTU) { cnt[tid] = 0; thr[tid] = 0ull; }

    // second-layer columns of this thread: two 4-wide groups (conflict-free 128-bit reads)
    const int colA = ct * 4, colB = C2P / 2 + ct * 4;

    for (int t0 = 0; t0 < p.n_items; t0 += kScTI) {
        __syncthreads();  // previous tile fully consumed; candidate lists settled
        for (int ul = warp; ul < kScTU; ul += kScThreads / 32)
            topk_make_room(cand, cnt, thr, cap, ul, p.k, lane);
        for (int e = tid; e < kScTI * (c1 / 4); e += kScThreads) {
            const int it = e / (c1 / 4), k4 = e % (c1 / 4);
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (t0 + it < p.n_items) v = ldg4(p.Q + (int64_t)(t0 + it) * p.ldq + k4 * 4);
            Qs[(k4 * 4 + 0) * kScQS + it] = v.x;
            Qs[(k4 * 4 + 1) * kScQS + it] = v.y;
            Qs[(k4 * 4 + 2) * kScQS + it] = v.z;
            Qs[(k4 * 4 + 3) * kScQS + it] = v.w;
        }
        __syncthreads();

        for (int pass = 0; pass < kScTU / UPP; ++pass) {
            const int ul = pass * UPP + user_in_pass;
            const float *pu = Ps + ul * c1;
            float acc[8][8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;
#pragma unroll 4
            for (int kk = 0; kk < c1; ++kk) {
                const float pv = pu[kk];
                const float4 q0 = *reinterpret_cast<const float4 *>(Qs + kk * kScQS + item_oct * 8);
                const float4 q1 = *reinterpret_cast<const float4 *>(Qs + kk * kScQS + item_oct * 8 + 4);
                const float4 w0 = *reinterpret_cast<const float4 *>(Ws + kk * C2P + colA);
                const float4 w1 = *reinterpret_cast<const float4 *>(Ws + kk * C2P + colB);
                const float a[8] = {fmaxf(pv + q0.x, 0.f), fmaxf(pv + q0.y, 0.f), fmaxf(pv + q0.z, 0.f), fmaxf(pv + q0.w, 0.f),
                                    fmaxf(pv + q1.x, 0.f), fmaxf(pv + q1.y, 0.f), fmaxf(pv + q1.z, 0.f), fmaxf(pv + q1.w, 0.f)};
                const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[j][c] = fmaf(a[j], w[c], acc[j][c]);
            }
            // epilogue: second-layer bias + relu, output layer, reduce over the CT column threads
            float bb[8], ww[8];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                bb[c] = b2s[colA + c]; ww[c] = w3s[colA + c];
                bb[4 + c] = b2s[colB + c]; ww[4 + c] = w3s[colB + c];
            }
            float mine = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float s = 0.f;
#pragma unroll
                for (int c = 0; c < 8; ++c) s = fmaf(fmaxf(acc[j][c] + bb[c], 0.f), ww[c], s);
#pragma unroll
                for (int o = CT / 2; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, CT);
                if ((j % CT) == ct) mine = s;  // column thread j finishes pair j (CT = 16: threads 8..15 idle here)
            }
            if (ct < 8) {
                const int item = t0 + item_oct * 8 + ct;
                const int64_t user = u0 + ul;
                if (item < p.n_items && user < p.n_users)
                    topk_offer<kExcl>(cand, cnt, thr, cap, ul, 1.f / (1.f + expf(-(mine + b3))), item, user,
                                      p.excl_rowptr, p.excl_items);
            }
        }
    }
    __syncthreads();
    for (int ul = warp; ul < kScTU; ul += kScThreads / 32)
        topk_write<false>(cand, cnt, thr, cap, ul, p.k, lane, u0 + ul, p.n_users, p.ids_out, p.scores_out);
}

template <int CT>
static size_t score_smem_bytes(int c1, int k) {
    const int C2P = CT * 8;
    size_t f = (size_t)c1 * C2P + (size_t)kScTU * c1 + (size_t)c1 * kScQS + 2 * C2P;
    f = (f + 1) / 2 * 2;  // keep the 64-bit candidate lists 8-byte aligned
    return f * sizeof(float) + topk_lists_smem_bytes(kScTU, k) + 16;
}

template <int CT>
static int launch_score(const ScoreParams &p, cudaStream_t s) {
    // up to the 227 KB a CTA may have: the widest classifier (c1 = 256, c2 = 128) at k = 128 needs 217 KB
    return launch_catalog_scorer(score_catalog_kernel<CT, false>, score_catalog_kernel<CT, true>, p,
                                 (unsigned)cdiv(p.n_users, kScTU), kScThreads, score_smem_bytes<CT>(p.c1, p.k), 227 * 1024,
                                 s, "score_catalog", "score_catalog");
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_score_catalog_topk(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                       int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                       const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                                       void *stream) {
    return cbrs_score_catalog_topk_ex(P, ldp, Q, ldq, n_users, n_items, c1, w2, b2, c2, w3, b3, k, ids_out, scores_out,
                                      nullptr, nullptr, stream);
}

extern "C" int cbrs_score_catalog_topk_ex(const float *P, int64_t ldp, const float *Q, int64_t ldq, int64_t n_users,
                                          int32_t n_items, int32_t c1, const float *w2, const float *b2, int32_t c2,
                                          const float *w3, const float *b3, int32_t k, int32_t *ids_out, float *scores_out,
                                          const int64_t *excl_rowptr, const int32_t *excl_items, void *stream) {
    CBRS_REQUIRE(P && Q && w2 && b2 && w3 && b3 && ids_out && scores_out, CBRS_E_INVALID, "score_catalog: null argument");
    const int rc = check_catalog_args("score_catalog", excl_rowptr, excl_items, n_users, n_items, k);
    if (rc != CBRS_OK) return rc;
    CBRS_REQUIRE(c1 > 0 && c1 % 4 == 0 && c1 <= 256 && c2 > 0 && c2 <= 128, CBRS_E_UNSUPPORTED,
                 "score_catalog: classifier widths c1=%d (multiple of 4, <= 256), c2=%d (<= 128)", c1, c2);
    CBRS_REQUIRE(ldp >= c1 && ldq >= c1 && ldq % 4 == 0 && ((uintptr_t)Q % 16) == 0, CBRS_E_INVALID,
                 "score_catalog: Q must be 16-byte aligned with ldq %% 4 == 0");
    if (n_users == 0) return CBRS_OK;
    ScoreParams p{P, ldp, Q, ldq, n_users, n_items, c1, c2, w2, b2, w3, b3, k, ids_out, scores_out, excl_rowptr, excl_items};
    return c2 <= 64 ? launch_score<8>(p, (cudaStream_t)stream) : launch_score<16>(p, (cudaStream_t)stream);
}
