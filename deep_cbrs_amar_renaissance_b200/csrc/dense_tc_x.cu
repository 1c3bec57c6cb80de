// Second tensor-core Dense kernel (see dense_tc.cu): cbrs_dense_tc uses it for deep layers (f1 + f2 >= 512, e.g. the
// hybrid scorer's 768 -> 256 BERT tower: 1.54 ms per 2^20 rows against 1.65 ms with dense_tc_kernel,
// profiles/r02_dense_tc_bench_variant4.jsonl).  tests/test_zz_gpu_dense_tc.py runs its parity cases at both depths and
// checks which kernel each depth gets.
// Written from the ncu evidence on dense_tc_kernel (profiles/r01_ncu_dense_tc_v3_stalls.txt: 8 warps per SM, ~535
// instructions per warp and K block, 26 % of the stall samples on the row-pointer LDS -> address arithmetic chain).
//
// Differences from dense_tc_kernel:
//   * 256 threads per CTA (16 warps per SM at 2 CTAs): a thread owns 4 (row, chunk) pairs instead of 8;
//   * a thread's chunk column c = tid & 7 never changes, so its 4 row pointers (per source) and its 4 swizzled
//     shared-memory offsets live in registers for the whole kernel, and the source selection (source 1 / source 2 /
//     zero padding) is one uniform decision per thread and K block: no LDS and no per-chunk predicates in the loop;
//   * the epilogue is split over the 8 warps: warp w reads TMEM lane quadrant w & 3 (the only one it may access) and
//     every second 16-column group (group parity = w >> 2).
#include "dense_tc.cuh"

namespace cbrs {

constexpr int kXThreads = 256;

__global__ void __launch_bounds__(kXThreads, 2) dense_tc_x_kernel(const __grid_constant__ DenseTcParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const int n_pad = (p.n + 15) / 16 * 16;
    const int k_total = p.f1 + p.f2;
    const int kb_count = (k_total + kDtKB - 1) / kDtKB;
    const int b_bytes = n_pad * 128;
    unsigned char *As = smem_raw;                          // [2][128][128 B]
    unsigned char *Bs = As + 2 * 16384;                    // [2][n_pad][128 B]
    uint64_t *mma_done = reinterpret_cast<uint64_t *>(Bs + 2 * b_bytes);   // [2]
    uint64_t *b_full = mma_done + 2;                                         // [2]
    float *bias_s = reinterpret_cast<float *>(b_full + 2);                   // [n_pad]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bias_s + n_pad);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
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
    // loop-invariant per thread: chunk column c, rows it*32 + (tid >> 3), their source pointers and tile offsets
    const int c = tid & 7;
    const float *rp1[4], *rp2[4];
    uint32_t soff[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int r = it * 32 + (tid >> 3);
        const int64_t m = (m0 + r < p.m) ? m0 + r : p.m - 1;   // rows past m read row m-1 again; never written out
        rp1[it] = p.x1 + (p.idx1 ? __ldg(p.idx1 + m) : m) * p.ld1;
        rp2[it] = p.x2 ? p.x2 + (p.idx2 ? __ldg(p.idx2 + m) : m) * p.ld2 : p.x1;
        soff[it] = tc::sw128_offset(r, c);
    }
    for (int e = tid; e < n_pad; e += kXThreads) bias_s[e] = (p.b && e < p.n) ? __ldg(p.b + e) : 0.f;
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t a_addr = tc::smem_u32(As), b_addr = tc::smem_u32(Bs);
    if ((a_addr & 1023u) != 0u) __trap();
    const uint32_t idesc = tc::idesc_bf16_f32(kDtRows, n_pad);
    const uint32_t zero_rt = (uint32_t)p.n >> 20;   // 0 at run time, unknown to the compiler (scheduling fence, see dense_tc.cu)

    auto issue = [&](int kb, float4 (&v)[8]) {
        const int kk = kb * kDtKB + c * 8;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const float *src = kk < p.f1 ? rp1[it] + kk : (kk < k_total ? rp2[it] + (kk - p.f1) : p.x1);
            v[2 * it] = dt_ld_stream4(src);
            v[2 * it + 1] = dt_ld_stream4(src + 4);
        }
    };
    auto finish = [&](int kb, float4 (&v)[8]) {
        unsigned char *a = As + (kb & 1) * 16384;
        const bool pad = kb * kDtKB + c * 8 >= k_total;
        uint32_t z = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) z ^= __float_as_uint(v[j].x);
        z &= zero_rt;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const float4 v0 = v[2 * it], v1 = v[2 * it + 1];
            uint4 packed = make_uint4(tc::pack_bf16x2(dt_or(v0.x, z), v0.y), tc::pack_bf16x2(dt_or(v0.z, z), v0.w),
                                      tc::pack_bf16x2(dt_or(v1.x, z), v1.y), tc::pack_bf16x2(dt_or(v1.z, z), v1.w));
            if (pad) packed = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4 *>(a + soff[it]) = packed;
        }
    };
    auto block = [&](int kb, float4 (&cur)[8], float4 (&nxt)[8]) {
        const int buf = kb & 1, use = kb >> 1;
        if (use > 0) {
            tc::mbar_wait(mma_done + buf, (uint32_t)(use - 1) & 1u);
            tc::tc_fence_after_sync();
        }
        if (warp == 0 && tc::elect_one()) {
            dt_expect_tx(b_full + buf, (uint32_t)b_bytes);
            const unsigned char *src = p.w_image + (size_t)kb * b_bytes;
            unsigned char *dst = Bs + buf * b_bytes;
            const int half = b_bytes / 2;
            dt_bulk_g2s(dst, src, (uint32_t)half, b_full + buf);
            dt_bulk_g2s(dst + half, src + half, (uint32_t)half, b_full + buf);
        }
        if (kb + 1 < kb_count) issue(kb + 1, nxt);
        finish(kb, cur);
        tc::fence_proxy_async_smem();
        tc::tc_fence_before_sync();
        __syncthreads();
        if (warp == 0 && tc::elect_one()) {
            tc::mbar_wait(b_full + buf, (uint32_t)use & 1u);
            tc::tc_fence_after_sync();
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const uint32_t koff = (uint32_t)s * 32;
                tc::mma_bf16_ss(tmem_base, tc::smem_desc_sw128(a_addr + buf * 16384 + koff),
                                tc::smem_desc_sw128(b_addr + buf * b_bytes + koff), idesc, (kb > 0 || s > 0) ? 1u : 0u);
            }
            tc::mma_commit(mma_done + buf);
        }
    };
    {
        float4 va[8], vb[8];
        issue(0, va);
        for (int kb = 0; kb < kb_count; kb += 2) {
            block(kb, va, vb);
            if (kb + 1 < kb_count) block(kb + 1, vb, va);
        }
    }
    tc::mbar_wait(mma_done + ((kb_count - 1) & 1), (uint32_t)((kb_count - 1) >> 1) & 1u);
    tc::tc_fence_after_sync();

    // ---- epilogue: warp w -> TMEM lane quadrant w & 3, 16-column groups of parity w >> 2 ----
    const int quad = warp & 3, parity = warp >> 2;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(quad * 32) << 16);
    const int64_t m = m0 + quad * 32 + lane;
    float *orow = p.out + (m < p.m ? m : 0) * p.ldo;
    const bool vec_ok = (p.ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15u) == 0);
    for (int cb = 0; cb < n_pad; cb += 16) {
        if (((cb >> 4) & 1) != parity) continue;     // uniform per warp: the tcgen05.ld below stays warp-collective
        uint32_t v[16];
        tc::tmem_ld16(tmem_row + (uint32_t)cb, v);
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

int dense_tc_launch_x(const DenseTcParams &p, cudaStream_t stream) {
    const int n_pad = (p.n + 15) / 16 * 16;
    const size_t smem = 2 * 16384 + 2 * (size_t)n_pad * 128 + 4 * sizeof(uint64_t) + (size_t)n_pad * 4 + 16;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(dense_tc_x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "cbrs_dense_tc (variant 4): %s", cudaGetErrorString(e));
        attr_set = true;
    }
    dense_tc_x_kernel<<<(unsigned)cdiv(p.m, kDtRows), kXThreads, smem, stream>>>(p);
    CBRS_CHECK_LAUNCH("cbrs_dense_tc (variant 4)");
    return CBRS_OK;
}

}  // namespace cbrs
