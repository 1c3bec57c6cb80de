// Shared between the tensor-core Dense kernels (dense_tc.cu: shallow layers; dense_tc_x.cu: deep layers, f1 + f2 >= 512).
#pragma once
#include "common.cuh"
#include "tc05.cuh"

namespace cbrs {

constexpr int kDtThreads = 128;
constexpr int kDtRows = 128;   // output rows per CTA = MMA M
constexpr int kDtKB = 64;      // K elements per block = one 128-byte swizzle row

struct DenseTcParams {
    const float *x1; int64_t ld1; const int64_t *idx1; int32_t f1;
    const float *x2; int64_t ld2; const int64_t *idx2; int32_t f2;
    const uint8_t *w_image;   // [kb][n_pad][128 B] bf16, SWIZZLE_128B
    const float *b;
    int64_t m; int32_t n; int32_t act;
    float *out; int64_t ldo;
};

__device__ __forceinline__ float dt_act(float v, int act) {
    switch (act) {
        case CBRS_ACT_RELU: return fmaxf(v, 0.f);
        case CBRS_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        case CBRS_ACT_TANH: return tanhf(v);
        default: return v;
    }
}

// 1-D bulk copy global -> shared through the async proxy (TMA engine), completion counted in bytes on an mbarrier
__device__ __forceinline__ void dt_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void dt_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ float dt_or(float v, uint32_t z) { return __uint_as_float(__float_as_uint(v) | z); }
__device__ __forceinline__ float4 dt_ld_stream4(const float *p) {   // read-once rows: keep them out of L1
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// deep-layer kernel (dense_tc_x.cu): cbrs_dense_tc runs it when f1 + f2 >= 512
int dense_tc_launch_x(const DenseTcParams &p, cudaStream_t stream);

}  // namespace cbrs
