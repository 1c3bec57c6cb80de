// bf16 tensor-core Dense layer (tcgen05 / TMEM), sm_100a: the GEMMs of the scorer towers
// (/root/reference/src/models/hybrid.py:74-77: Dense 768 -> 256 -> 64 over the BERT rows; models/basic.py:33-34).
//
//   out[m, 0:n] = act( bf16([ X1[idx1[m], 0:f1] || X2[idx2[m], 0:f2] ]) @ bf16(W[f1+f2, n]) + b ),  fp32 accumulate
//
// Same contract as cbrs_dense (dense.cu: fused gather + concat + bias + activation, Keras kernel layout) with the
// product on the 5th-generation tensor cores.  One CTA owns 128 output rows:
//   * K is walked in blocks of 64.  For every block the 128 threads build the A operand tile - 128 rows x 64 bf16 in
//     the canonical K-major SWIZZLE_128B layout - straight from the fp32 rows in HBM (8 threads per row, 32 B of fp32
//     each, so a warp reads four 256-byte row segments: coalesced; a thread's 16 loads are all in flight before the
//     first is used) while one cp.async.bulk brings the matching block of the pre-swizzled bf16 image of W
//     (cbrs_dense_tc_prepare) next to it, counted on an mbarrier the MMA-issuing thread waits on;
//   * one thread issues four tcgen05.mma (M=128, N=n_pad, K=16) per block into ONE TMEM accumulator and commits to the
//     block's mbarrier; tiles are double buffered, so the tensor core works on block b while the CTA builds b+1, and
//     the fp32 rows of block b+1 are already on their way into a second register set while block b is converted;
//   * thread t reads accumulator row t back with tcgen05.ld (warp w owns TMEM lanes 32w..32w+31), adds the bias,
//     applies the activation and writes its fp32 output row.
// HBM-side the kernel reads every A row once (fp32) and W once per CTA (L2 resident: <= 393 KB at 768 x 256).
// Precision: operands rounded to bf16 (nearest even), products and sums fp32 - the parity tests compare against an
// oracle that rounds the same operands (tolerance stated there); the fp32 FFMA kernel stays the 1e-5 parity path.
#include "dense_tc.cuh"

#include <algorithm>

namespace cbrs {

// W [k, n] fp32 (Keras [in,out]) -> B operand image: element (col, kk) = bf16(W[kk][col]), K-major, SWIZZLE_128B,
// zero padded to n_pad columns and kb_count * 64 rows of K
__global__ void dense_tc_prep_kernel(const float *__restrict__ w, int k, int n, int n_pad, int kb_count,
                                     uint8_t *__restrict__ image) {
    const int64_t total = (int64_t)kb_count * n_pad * kDtKB;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int kb = (int)(e / (n_pad * kDtKB)), rem = (int)(e % (n_pad * kDtKB));
        const int col = rem % n_pad, kk = rem / n_pad;   // consecutive threads read consecutive columns of one W row
        const int kg = kb * kDtKB + kk;
        const float v = (col < n && kg < k) ? w[(int64_t)kg * n + col] : 0.f;
        const uint32_t off = (uint32_t)kb * n_pad * 128 + tc::sw128_offset(col, kk >> 3) + (kk & 7) * 2;
        *reinterpret_cast<__nv_bfloat16 *>(image + off) = __float2bfloat16_rn(v);
    }
}

__global__ void __launch_bounds__(kDtThreads, 2) dense_tc_kernel(const __grid_constant__ DenseTcParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];  // SWIZZLE_128B tiles need 1024-byte alignment
    const int n_pad = (p.n + 15) / 16 * 16;
    const int k_total = p.f1 + p.f2;
    const int kb_count = (k_total + kDtKB - 1) / kDtKB;
    const int b_bytes = n_pad * 128;
    unsigned char *As = smem_raw;                          // [2][128][128 B]
    unsigned char *Bs = As + 2 * 16384;                    // [2][n_pad][128 B]
    const float **row1 = reinterpret_cast<const float **>(Bs + 2 * b_bytes);   // [128] start of the row in source 1
    const float **row2 = row1 + kDtRows;                                          // [128] ... in source 2
    uint64_t *mma_done = reinterpret_cast<uint64_t *>(row2 + kDtRows);            // [2] MMAs that read buffer b completed
    uint64_t *b_full = mma_done + 2;                                              // [2] bulk copy of the B tile landed
    float *bias_s = reinterpret_cast<float *>(b_full + 2);                        // [n_pad]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bias_s + n_pad);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int64_t m0 = (int64_t)blockIdx.x * kDtRows;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < n_pad) tmem_cols <<= 1;

    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 0) {
        tc::mbar_init(mma_done, 1);
        tc::mbar_init(mma_done + 1, 1);
        tc::mbar_init(b_full, 1);
        tc::mbar_init(b_full + 1, 1);
        tc::fence_mbar_init();
    }
    {   // gather indices are resolved once per row: pointer to the row's first element in each source.  Rows past m
        // read row m-1 again (valid memory; their accumulator rows are never written out)
        const int64_t m = (m0 + tid < p.m) ? m0 + tid : p.m - 1;
        row1[tid] = p.x1 + (p.idx1 ? __ldg(p.idx1 + m) : m) * p.ld1;
        row2[tid] = p.x2 ? p.x2 + (p.idx2 ? __ldg(p.idx2 + m) : m) * p.ld2 : p.x1;
        for (int e = tid; e < n_pad; e += kDtThreads) bias_s[e] = (p.b && e < p.n) ? __ldg(p.b + e) : 0.f;
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);  // this warp's lane quadrant
    const uint32_t a_addr = tc::smem_u32(As), b_addr = tc::smem_u32(Bs);
    if ((a_addr & 1023u) != 0u) __trap();  // the runtime honours the declared alignment; fail loudly if not
    const uint32_t idesc = tc::idesc_bf16_f32(kDtRows, n_pad);
    const uint32_t zero_rt = (uint32_t)p.n >> 20;   // 0 (n <= 256), but not to the compiler: see finish()

    // A tile of block kb: 128 rows x 8 chunks of 8 bf16; thread -> (row, chunk), 8 consecutive threads per row.
    // issue(): all 16 loads of the thread (two float4 per chunk) go out back to back.
    auto issue = [&](int kb, float4 (&v)[16]) {
        const float *src[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int e = it * kDtThreads + tid;
            const int r = e >> 3, c = e & 7;
            const int kk = kb * kDtKB + c * 8;      // f1 and f2 are multiples of 8: a chunk never straddles the sources
            src[it] = kk >= k_total ? p.x1 : (kk < p.f1 ? row1[r] + kk : row2[r] + (kk - p.f1));
        }
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            v[2 * it] = dt_ld_stream4(src[it]);
            v[2 * it + 1] = dt_ld_stream4(src[it] + 4);
        }
    };
    // finish(): convert to bf16 and store in operand layout.  Scheduling fence: ptxas otherwise interleaves conversions
    // with the loads and each pair of loads waits for the previous pair's round trip - one operand of every conversion
    // ORs in a (run-time) zero derived from ALL 16 loads, so no conversion is scheduled before every load was issued.
    auto finish = [&](int kb, float4 (&v)[16]) {
        unsigned char *a = As + (kb & 1) * 16384;
        uint32_t z = 0u;
#pragma unroll
        for (int j = 0; j < 16; ++j) z ^= __float_as_uint(v[j].x);
        z &= zero_rt;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int e = it * kDtThreads + tid;
            const int r = e >> 3, c = e & 7;
            const float4 v0 = v[2 * it], v1 = v[2 * it + 1];
            uint4 packed = make_uint4(tc::pack_bf16x2(dt_or(v0.x, z), v0.y), tc::pack_bf16x2(dt_or(v0.z, z), v0.w),
                                      tc::pack_bf16x2(dt_or(v1.x, z), v1.y), tc::pack_bf16x2(dt_or(v1.z, z), v1.w));
            if (kb * kDtKB + c * 8 >= k_total) packed = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4 *>(a + tc::sw128_offset(r, c)) = packed;
        }
    };
    // one K block: B tile by bulk copy, prefetch of the NEXT block's A rows into the other register set (their round
    // trip overlaps this block's conversion, barrier and MMA issue), conversion of this block, MMAs
    auto block = [&](int kb, float4 (&cur)[16], float4 (&nxt)[16]) {
        const int buf = kb & 1, use = kb >> 1;
        if (use > 0) {  // the MMAs that read this buffer pair two blocks ago must have completed
            tc::mbar_wait(mma_done + buf, (uint32_t)(use - 1) & 1u);
            tc::tc_fence_after_sync();
        }
        if (warp == 0 && tc::elect_one()) {   // block kb of the image (already in operand layout); lands while A is being built
            dt_expect_tx(b_full + buf, (uint32_t)b_bytes);
            const unsigned char *src = p.w_image + (size_t)kb * b_bytes;
            unsigned char *dst = Bs + buf * b_bytes;
            const int half = b_bytes / 2;   // n_pad * 64: a multiple of 16 bytes, at most 16 KB per copy
            dt_bulk_g2s(dst, src, (uint32_t)half, b_full + buf);
            dt_bulk_g2s(dst + half, src + half, (uint32_t)half, b_full + buf);
        }
        if (kb + 1 < kb_count) issue(kb + 1, nxt);
        finish(kb, cur);
        tc::fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core
        tc::tc_fence_before_sync();
        __syncthreads();
        if (warp == 0 && tc::elect_one()) {   // elected: UTCHMMA issues once, not in a per-lane loop
            tc::mbar_wait(b_full + buf, (uint32_t)use & 1u);
            tc::tc_fence_after_sync();
#pragma unroll
            for (int s = 0; s < 4; ++s) {           // 4 x K=16 inside the 64-wide block (zero padded past k_total)
                const uint32_t koff = (uint32_t)s * 32;
                tc::mma_bf16_ss(tmem_base, tc::smem_desc_sw128(a_addr + buf * 16384 + koff),
                                tc::smem_desc_sw128(b_addr + buf * b_bytes + koff), idesc, (kb > 0 || s > 0) ? 1u : 0u);
            }
            tc::mma_commit(mma_done + buf);
        }
    };
    {
        float4 va[16], vb[16];
        issue(0, va);
        for (int kb = 0; kb < kb_count; kb += 2) {
            block(kb, va, vb);
            if (kb + 1 < kb_count) block(kb + 1, vb, va);
        }
    }
    // the last commit covers every MMA issued before it (and every bulk copy was waited for before its MMAs)
    tc::mbar_wait(mma_done + ((kb_count - 1) & 1), (uint32_t)((kb_count - 1) >> 1) & 1u);
    tc::tc_fence_after_sync();

    // ---- epilogue: accumulator row `tid` -> bias, activation, fp32 row ----
    const int64_t m = m0 + tid;
    float *orow = p.out + (m < p.m ? m : 0) * p.ldo;
    const bool vec_ok = (p.ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15u) == 0);
    for (int cb = 0; cb < n_pad; cb += 16) {
        uint32_t v[16];
        tc::tmem_ld16(tmem_row + (uint32_t)cb, v);   // warp-collective: executed by every thread
        tc::tmem_ld_wait();
        if (m < p.m) {
            float o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = dt_act(__uint_as_float(v[j]) + bias_s[cb + j], p.act);
            if (vec_ok && cb + 16 <= p.n) {
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4 *>(orow + cb + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (cb + j < p.n) orow[cb + j] = o[j];
            }
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, tmem_cols);
    }
}

static size_t dense_tc_smem_bytes(int n_pad) {
    return 2 * 16384 + 2 * (size_t)n_pad * 128 + 2 * kDtRows * sizeof(void *) + 4 * sizeof(uint64_t) + (size_t)n_pad * 4 + 16;
}

}  // namespace cbrs

using namespace cbrs;

extern "C" size_t cbrs_dense_tc_image_bytes(int32_t k, int32_t n) {
    if (k <= 0 || n <= 0) return 0;
    const size_t n_pad = (size_t)(n + 15) / 16 * 16, kb = (size_t)(k + kDtKB - 1) / kDtKB;
    return kb * n_pad * 128;
}

extern "C" int cbrs_dense_tc_prepare(const float *w, int32_t k, int32_t n, void *image, void *stream) {
    CBRS_REQUIRE(w && image, CBRS_E_INVALID, "cbrs_dense_tc_prepare: null pointer");
    CBRS_REQUIRE(k > 0 && n > 0 && n <= 256, CBRS_E_INVALID, "cbrs_dense_tc_prepare: k = %d, n = %d (1 <= n <= 256)", k, n);
    CBRS_REQUIRE((reinterpret_cast<uintptr_t>(image) & 15u) == 0, CBRS_E_INVALID, "cbrs_dense_tc_prepare: image must be 16-byte aligned");
    const int n_pad = (n + 15) / 16 * 16, kb = (k + kDtKB - 1) / kDtKB;
    const int64_t total = (int64_t)kb * n_pad * kDtKB;
    const int blocks = (int)std::min<int64_t>(cdiv(total, 256), 4 * kSMs);
    dense_tc_prep_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, k, n, n_pad, kb, (uint8_t *)image);
    CBRS_CHECK_LAUNCH("cbrs_dense_tc_prepare");
    return CBRS_OK;
}

extern "C" int cbrs_dense_tc(const float *x1, int64_t ld1, const int64_t *idx1, int32_t f1, const float *x2, int64_t ld2,
                             const int64_t *idx2, int32_t f2, const void *w_image, const float *b, int64_t m, int32_t n,
                             int act, float *out, int64_t ldo, void *stream) {
    CBRS_REQUIRE(x1 && w_image && out, CBRS_E_INVALID, "cbrs_dense_tc: null pointer");
    CBRS_REQUIRE(m >= 0 && n > 0 && n <= 256, CBRS_E_INVALID, "cbrs_dense_tc: n = %d (1 <= n <= 256; wider layers: cbrs_dense)", n);
    CBRS_REQUIRE(f1 > 0 && f1 % 8 == 0 && f2 >= 0 && f2 % 8 == 0, CBRS_E_INVALID,
                 "cbrs_dense_tc: source widths must be multiples of 8 (f1 = %d, f2 = %d)", f1, f2);
    CBRS_REQUIRE((f2 == 0) == (x2 == nullptr), CBRS_E_INVALID, "cbrs_dense_tc: x2 and f2 disagree");
    CBRS_REQUIRE(ld1 % 4 == 0 && (reinterpret_cast<uintptr_t>(x1) & 15u) == 0 &&
                     (!x2 || (ld2 % 4 == 0 && (reinterpret_cast<uintptr_t>(x2) & 15u) == 0)),
                 CBRS_E_INVALID, "cbrs_dense_tc: source rows must be 16-byte aligned (ld %% 4 == 0)");
    CBRS_REQUIRE(act >= CBRS_ACT_NONE && act <= CBRS_ACT_TANH, CBRS_E_INVALID, "cbrs_dense_tc: unknown activation %d", act);
    CBRS_REQUIRE(ldo >= n, CBRS_E_INVALID, "cbrs_dense_tc: ldo < n");
    if (m == 0) return CBRS_OK;
    const int n_pad = (n + 15) / 16 * 16;
    const size_t smem = dense_tc_smem_bytes(n_pad);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(dense_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 101 * 1024);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "cbrs_dense_tc: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    DenseTcParams p;
    p.x1 = x1; p.ld1 = ld1; p.idx1 = idx1; p.f1 = f1;
    p.x2 = x2; p.ld2 = ld2; p.idx2 = idx2; p.f2 = f2;
    p.w_image = (const uint8_t *)w_image; p.b = b; p.m = m; p.n = n; p.act = act; p.out = out; p.ldo = ldo;
    // two kernels, chosen by depth (profiles/r02_dense_tc_bench_{shipped,variant4}.jsonl, 2^20 rows): the 256-thread
    // kernel with loop-invariant row pointers (dense_tc_x.cu) wins on deep layers (768 -> 256: 1.54 vs 1.65 ms), the
    // 128-thread one on shallow layers (256 -> 64: 0.34 vs 0.40 ms).
    if (f1 + f2 >= 512) return dense_tc_launch_x(p, (cudaStream_t)stream);
    dense_tc_kernel<<<(unsigned)cdiv(m, kDtRows), kDtThreads, smem, (cudaStream_t)stream>>>(p);
    CBRS_CHECK_LAUNCH("cbrs_dense_tc");
    return CBRS_OK;
}
