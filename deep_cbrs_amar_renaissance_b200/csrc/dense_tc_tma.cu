// bf16 tensor-core Dense layer fed by TMA from bf16-STORED sources (tcgen05 / TMEM / cp.async.bulk.tensor), sm_100a:
// the tower GEMMs of the hybrid scorer over the static content table
// (/root/reference/src/models/hybrid.py:74-77: Dense 768 -> 256 -> 64 over the BERT rows, gathered by the batch's ids at
// hybrid.py:136-140).
//
//   out[m, 0:n] = act( [ X1[idx1[m], 0:f1] || X2[idx2[m], 0:f2] ] @ bf16(W[f1+f2, n]) + b ),  X1, X2 bf16, fp32 accumulate
//
// dense_tc.cu reads fp32 rows and converts them in registers on every call (0.40-0.43 of the HBM roofline at 768 -> 256,
// 8 warps per SM busy building operand tiles).  The content table is static, so it is rounded to bf16 ONCE
// (cbrs_convert_f32_bf16 - the same round-to-nearest-even the fp32 kernel applies per call, so both kernels multiply the
// same operands) and this kernel never touches a row with a thread:
//   warps 0-3 producers, 64 rows of the tile each.  Per K block of 64 (one 128-byte swizzle row): the A operand - 256 rows x
//             128 B - lands straight in the canonical K-major SWIZZLE_128B layout, by one tiled cp.async.bulk.tensor.2d
//             per warp when the rows are consecutive, or by 16 tile::gather4 loads per warp (4 indexed rows each, one
//             per lane 0-15: UTMALDG takes its coordinates from uniform registers, so the compiler issues them lane by
//             lane - hence four warps) when they are gathered; one cp.async.bulk brings the matching block of the
//             pre-swizzled image of W (cbrs_dense_tc_prepare).  A ring of 3-6 such stages (64 KB each at n = 256)
//             keeps ~190 KB per SM in flight.
//   warp 4    one thread issues 4 x 2 tcgen05.mma (M=128, N=n_pad, K=16) per stage: TWO 128-row accumulators share every
//             W block, which halves the L2 -> SM traffic of W (393 KB per pass at 768 x 256 - more than the rows
//             themselves); the commit of a stage's MMAs returns the stage to the producer.
//   warps 5-12 epilogue: tcgen05.ld (warp w owns TMEM lanes 32 (w % 4)..; warps 5-8 drain accumulator 0, warps 9-12
//             accumulator 1), bias, activation, a turn through a 4 KB staging buffer per warp so that global stores are
//             4 full rows x 128 B per instruction, fp32 or bf16 output.  For n <= 128 the accumulator pair
//             is double buffered in TMEM, so the next tile's MMAs run under the epilogue; at n = 256 the pair fills
//             all 512 columns and the ring absorbs the epilogue instead (the producer keeps loading).
// One persistent CTA per SM, static tile schedule.  HBM traffic: every source row once as bf16 + the output once.
#include "common.cuh"
#include "tc05.cuh"

#include <cuda.h>  // CUtensorMap; the encoder is looked up through the runtime (no -lcuda)

namespace cbrs {

constexpr int kTmRows = 256;               // output rows per tile: two MMA M=128 halves
constexpr int kTmKB = 64;                  // bf16 elements per 128-byte swizzle row = K per stage
constexpr int kTmABytes = kTmRows * 128;   // A operand of one stage
constexpr int kTmThreads = 416;             // 4 producer warps, the MMA warp, 8 epilogue warps
constexpr int kTmProducers = 4;            // producer warps, 64 rows of the tile each
constexpr int kTmMaxStages = 6;
constexpr int kTmStaging = 8 * 4096;       // epilogue staging: 4 KB per epilogue warp

struct TmParams {
    const int64_t *idx1, *idx2;
    int32_t kb1, kb2;          // K blocks taken from source 1 / source 2
    int32_t gather1, gather2;  // source rows are indexed (tile::gather4) / consecutive (tiled box)
    const uint8_t *w_image;    // [kb][n_pad][128 B] bf16, SWIZZLE_128B (cbrs_dense_tc_prepare)
    const float *b;
    int64_t m;
    int32_t n, n_pad, act;
    void *out;
    int64_t ldo;
    int32_t out_bf16;
    int64_t n_tiles;
    int32_t stages, acc_sets;
};

__device__ __forceinline__ float tm_act(float v, int act) {
    switch (act) {
        case CBRS_ACT_RELU: return fmaxf(v, 0.f);
        case CBRS_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        case CBRS_ACT_TANH: return tanhf(v);
        default: return v;
    }
}
__device__ __forceinline__ void tm_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tm_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tm_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
                 : "memory");
}
// tiled 2-D load: box (64 columns, 64 rows) at (col, row); rows past the tensor arrive as zeros
__device__ __forceinline__ void tm_tma_tile(void *dst, const CUtensorMap *map, int32_t col, int32_t row, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            tc::smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(col), "r"(row), "r"(tc::smem_u32(bar))
        : "memory");
}
// four indexed rows (box 64 columns x 1 row each) -> four consecutive 128-byte rows of the operand tile
__device__ __forceinline__ void tm_tma_gather4(void *dst, const CUtensorMap *map, int32_t col, int32_t r0, int32_t r1, int32_t r2,
                                               int32_t r3, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], "
        "[%7];" ::"r"(tc::smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(col), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(tc::smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tm_st4(float *p, float a, float b, float c, float d) {
    *reinterpret_cast<float4 *>(p) = make_float4(a, b, c, d);
}

__global__ void convert_f32_bf16_kernel(const float *__restrict__ x, int64_t ldx, int64_t m, int k, __nv_bfloat16 *__restrict__ out,
                                        int64_t ldo) {
    const int64_t total = m * (int64_t)(k / 4);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / (k / 4);
        const int c = (int)(e % (k / 4)) * 4;
        const float4 v = *reinterpret_cast<const float4 *>(x + r * ldx + c);
        uint2 w = make_uint2(tc::pack_bf16x2(v.x, v.y), tc::pack_bf16x2(v.z, v.w));
        *reinterpret_cast<uint2 *>(out + r * ldo + c) = w;
    }
}

template <int kAct>
__device__ __forceinline__ float tm_act_c(float v) {
    if (kAct == CBRS_ACT_RELU) return fmaxf(v, 0.f);
    if (kAct == CBRS_ACT_SIGMOID) return 1.f / (1.f + expf(-v));
    if (kAct == CBRS_ACT_TANH) return tanhf(v);
    return v;
}

// Epilogue of one warp (warps 5..12) over all tiles of its CTA.
// A thread holds ONE accumulator row (TMEM lane), so storing it directly writes 16 bytes to 32 different lines per
// instruction.  Each warp turns its 32 x 32 block through a private 4 KB staging buffer instead (16-byte chunks
// XOR-swizzled by row: conflict-free both ways) and writes 4 rows x 128 contiguous bytes per instruction.
template <int kAct>
__device__ __forceinline__ void tm_epilogue(const TmParams &p, unsigned char *stg, const float *bias_s, uint64_t *acc_full,
                                            uint64_t *acc_empty, uint32_t tmem_base, int64_t my_tiles) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int quad = warp & 3;              // TMEM lane quadrant this warp may read
    const int half = (warp - kTmProducers - 1) >> 2;   // accumulator (row half) of the tile
    const bool vec_ok = p.out_bf16 ? (p.ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 7u) == 0)
                                   : (p.ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15u) == 0);
    const int rr = lane >> 3, c4 = lane & 7;   // read-back role: row rr of every group of 4 rows, 16-byte chunk c4
    for (int64_t lt = 0; lt < my_tiles; ++lt) {
        const int64_t tile = blockIdx.x + lt * gridDim.x;
        const int set = (int)(lt % p.acc_sets);
        tc::mbar_wait(acc_full + set, (uint32_t)(lt / p.acc_sets) & 1u);
        tc::tc_fence_after_sync();
        const int64_t row_base = tile * kTmRows + half * 128 + quad * 32;
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)((set * 2 + half) * p.n_pad);
        uint32_t v[32];
        auto load = [&](int cb) {   // warp-collective; a trailing 16-column block (n_pad % 32 == 16) loads half
            if (cb + 32 <= p.n_pad) {
                tc::tmem_ld32(taddr + (uint32_t)cb, v);
            } else {
                uint32_t h[16];
                tc::tmem_ld16(taddr + (uint32_t)cb, h);
#pragma unroll
                for (int j = 0; j < 16; ++j) { v[j] = h[j]; v[16 + j] = 0u; }
            }
        };
        load(0);
        for (int cb = 0; cb < p.n_pad; cb += 32) {
            tc::tmem_ld_wait();
            const bool last = cb + 32 >= p.n_pad;
            if (last) {   // every TMEM read of this tile has returned: the MMA warp may overwrite the accumulators
                tc::tc_fence_before_sync();
                tm_arrive(acc_empty + set);
            }
            const int ncol = last ? p.n_pad - cb : 32;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float4 o;
                const int c = cb + 4 * j;
                if (4 * j < ncol) {
                    const float4 bv = *reinterpret_cast<const float4 *>(bias_s + c);
                    o.x = tm_act_c<kAct>(__uint_as_float(v[4 * j]) + bv.x);
                    o.y = tm_act_c<kAct>(__uint_as_float(v[4 * j + 1]) + bv.y);
                    o.z = tm_act_c<kAct>(__uint_as_float(v[4 * j + 2]) + bv.z);
                    o.w = tm_act_c<kAct>(__uint_as_float(v[4 * j + 3]) + bv.w);
                    *reinterpret_cast<float4 *>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) = o;
                }
            }
            if (!last) load(cb + 32);   // in flight while this block is written out
            __syncwarp();
            const int col = cb + c4 * 4;
            if (c4 * 4 < ncol) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + rr;
                    const float4 o = *reinterpret_cast<const float4 *>(stg + r * 128 + ((c4 ^ (r & 7)) << 4));
                    const int64_t grow = row_base + r;
                    if (grow < p.m) {
                        if (p.out_bf16) {
                            __nv_bfloat16 *dst = reinterpret_cast<__nv_bfloat16 *>(p.out) + grow * p.ldo + col;
                            if (vec_ok && col + 4 <= p.n) {
                                *reinterpret_cast<uint2 *>(dst) = make_uint2(tc::pack_bf16x2(o.x, o.y), tc::pack_bf16x2(o.z, o.w));
                            } else {
                                const float e[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                                for (int t = 0; t < 4; ++t)
                                    if (col + t < p.n) dst[t] = __float2bfloat16_rn(e[t]);
                            }
                        } else {
                            float *dst = reinterpret_cast<float *>(p.out) + grow * p.ldo + col;
                            if (vec_ok && col + 4 <= p.n) {
                                *reinterpret_cast<float4 *>(dst) = o;
                            } else {
                                const float e[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                                for (int t = 0; t < 4; ++t)
                                    if (col + t < p.n) dst[t] = e[t];
                            }
                        }
                    }
                }
            }
            __syncwarp();   // the staging buffer is rewritten by the next block
        }
    }
}

__global__ void __launch_bounds__(kTmThreads, 1)
    dense_tc_tma_kernel(const __grid_constant__ CUtensorMap map1, const __grid_constant__ CUtensorMap map2,
                        const __grid_constant__ TmParams p) {
    extern __shared__ __align__(1024) unsigned char tm_smem[];
    const int w_bytes = p.n_pad * 128;                      // W operand of one stage
    const int stage_bytes = kTmABytes + w_bytes;
    unsigned char *ring = tm_smem;                          // [stages][A 32 KB | W n_pad * 128 B]
    unsigned char *staging = ring + (size_t)p.stages * stage_bytes;   // [8 epilogue warps][32 rows x 128 B]
    uint64_t *bars = reinterpret_cast<uint64_t *>(staging + kTmStaging);
    uint64_t *full = bars, *empty = bars + kTmMaxStages, *acc_full = empty + kTmMaxStages, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
    float *bias_s = reinterpret_cast<float *>(tmem_slot + 4);   // 16-byte aligned: read as float4

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kb_total = p.kb1 + p.kb2;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * p.acc_sets * p.n_pad) tmem_cols <<= 1;
    if ((tc::smem_u32(tm_smem) & 1023u) != 0u) __trap();   // SWIZZLE_128B tiles need the declared alignment

    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 32) {
        for (int s = 0; s < p.stages; ++s) {
            tc::mbar_init(full + s, kTmProducers);
            tc::mbar_init(empty + s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(acc_full + a, 1);
            tc::mbar_init(acc_empty + a, 256);
        }
        tc::fence_mbar_init();
    }
    for (int e = tid; e < p.n_pad; e += kTmThreads) bias_s[e] = (p.b && e < p.n) ? __ldg(p.b + e) : 0.f;
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t my_tiles = (p.n_tiles > (int64_t)blockIdx.x) ? (p.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp < kTmProducers) {
        // ---------------- producers: warp w feeds rows 64w..64w+63 of every tile ----------------
        const uint32_t my_bytes = 64 * 128 + (warp == 0 ? (uint32_t)w_bytes : 0u);   // what this warp adds to a stage
        int64_t it = 0;
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            const int64_t row0 = (blockIdx.x + lt * gridDim.x) * kTmRows + warp * 64;
            // lane l < 16 feeds rows 4l..4l+3 of the warp's 64; rows past m re-read row m-1 (valid memory, never written out)
            int32_t r1[4], r2[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int64_t r = row0 + (lane & 15) * 4 + j;
                if (r >= p.m) r = p.m - 1;
                r1[j] = p.gather1 ? (int32_t)__ldg(p.idx1 + r) : (int32_t)r;
                r2[j] = p.gather2 ? (int32_t)__ldg(p.idx2 + r) : (int32_t)r;
            }
            for (int kb = 0; kb < kb_total; ++kb, ++it) {
                const int s = (int)(it % p.stages);
                const int64_t use = it / p.stages;
                if (use > 0) tc::mbar_wait(empty + s, (uint32_t)(use - 1) & 1u);
                unsigned char *a_dst = ring + (size_t)s * stage_bytes + warp * (64 * 128);
                const bool first = kb < p.kb1;
                const bool gather = first ? p.gather1 : p.gather2;
                const CUtensorMap *map = first ? &map1 : &map2;
                const int32_t col = (first ? kb : kb - p.kb1) * kTmKB;
                if (lane == 0) {
                    tm_expect_tx(full + s, my_bytes);
                    if (warp == 0) {
                        const unsigned char *w_src = p.w_image + (size_t)kb * w_bytes;
                        unsigned char *w_dst = ring + (size_t)s * stage_bytes + kTmABytes;
                        for (int off = 0; off < w_bytes; off += 16384) {
                            const int nb = (w_bytes - off < 16384) ? w_bytes - off : 16384;
                            tm_bulk_g2s(w_dst + off, w_src + off, (uint32_t)nb, full + s);
                        }
                    }
                    if (!gather) tm_tma_tile(a_dst, map, col, (int32_t)row0, full + s);
                }
                __syncwarp();
                if (gather && lane < 16)
                    tm_tma_gather4(a_dst + (lane * 4) * 128, map, col, first ? r1[0] : r2[0], first ? r1[1] : r2[1],
                                   first ? r1[2] : r2[2], first ? r1[3] : r2[3], full + s);
            }
        }
    } else if (warp == kTmProducers) {
        // ---------------- MMA issuer ----------------
        if (tc::elect_one()) {   // one lane, and ptxas knows it: UTCHMMA issues once, not in a per-lane loop
            const uint32_t idesc = tc::idesc_bf16_f32(128, p.n_pad);
            const uint32_t ring_addr = tc::smem_u32(ring);
            int64_t it = 0;
            for (int64_t lt = 0; lt < my_tiles; ++lt) {
                const int set = (int)(lt % p.acc_sets);
                const int64_t set_use = lt / p.acc_sets;
                if (set_use > 0) tc::mbar_wait(acc_empty + set, (uint32_t)(set_use - 1) & 1u);
                tc::tc_fence_after_sync();
                const uint32_t d0 = tmem_base + (uint32_t)(set * 2 * p.n_pad), d1 = d0 + (uint32_t)p.n_pad;
                for (int kb = 0; kb < kb_total; ++kb, ++it) {
                    const int s = (int)(it % p.stages);
                    tc::mbar_wait(full + s, (uint32_t)(it / p.stages) & 1u);
                    tc::tc_fence_after_sync();
                    const uint32_t a0 = ring_addr + (uint32_t)s * stage_bytes, a1 = a0 + 128 * 128, bw = a0 + kTmABytes;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {   // 4 x K=16 inside the 64-wide block
                        const uint32_t koff = (uint32_t)ks * 32;
                        const uint64_t db = tc::smem_desc_sw128(bw + koff);
                        tc::mma_bf16_ss(d0, tc::smem_desc_sw128(a0 + koff), db, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
                        tc::mma_bf16_ss(d1, tc::smem_desc_sw128(a1 + koff), db, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
                    }
                    tc::mma_commit(empty + s);      // the stage is free once these MMAs have read it
                }
                tc::mma_commit(acc_full + set);     // both accumulators of the tile complete
            }
        }
    } else {
        // ---------------- epilogue (warps 5..12) ----------------
        unsigned char *stg = staging + (warp - kTmProducers - 1) * 4096;
        switch (p.act) {   // the activation is a compile-time constant of the loop (a per-element switch is ~3 branches each)
            case CBRS_ACT_RELU: tm_epilogue<CBRS_ACT_RELU>(p, stg, bias_s, acc_full, acc_empty, tmem_base, my_tiles); break;
            case CBRS_ACT_SIGMOID: tm_epilogue<CBRS_ACT_SIGMOID>(p, stg, bias_s, acc_full, acc_empty, tmem_base, my_tiles); break;
            case CBRS_ACT_TANH: tm_epilogue<CBRS_ACT_TANH>(p, stg, bias_s, acc_full, acc_empty, tmem_base, my_tiles); break;
            default: tm_epilogue<CBRS_ACT_NONE>(p, stg, bias_s, acc_full, acc_empty, tmem_base, my_tiles); break;
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, tmem_cols);
    }
}

static size_t tm_tail_bytes(int n_pad) { return kTmStaging + (2 * kTmMaxStages + 4) * sizeof(uint64_t) + 16 + (size_t)n_pad * 4 + 64; }
static int tm_stages(int n_pad) {
    const size_t stage = kTmABytes + (size_t)n_pad * 128;
    const size_t room = 227 * 1024 - tm_tail_bytes(n_pad);
    int s = (int)(room / stage);
    return s > kTmMaxStages ? kTmMaxStages : s;
}

typedef CUresult (*tm_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                 const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static tm_encode_fn tm_encoder() {
    static tm_encode_fn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (tm_encode_fn)ptr;
    }
    return fn;
}
// L2 promotion of the loads: a row is read in 128-byte slices, one K block at a time; promoting each miss to 256 B brings the
// next K block's slice of the same row along (measured, 768 -> 256 at 2^20 rows: 0.543 vs 0.558 ms consecutive, 0.609 vs
// 0.623 ms gathered, profiles/r02_dense_tc_tma_bench_l2p{128,256}.jsonl).
constexpr CUtensorMapL2promotion kTmL2Promotion = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
// rows of `f` bf16 out of a [rows, ld] table; box = 64 columns x (1 row for tile::gather4 | 64 rows tiled)
static int tm_make_map(CUtensorMap *map, const void *x, int64_t ld, int64_t rows, int32_t f, bool gather) {
    tm_encode_fn encode = tm_encoder();
    CBRS_REQUIRE(encode, CBRS_E_CUDA, "cbrs_dense_tc_bf16: cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[2] = {(cuuint64_t)f, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kTmKB, gather ? 1u : 64u};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(x), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, kTmL2Promotion,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CBRS_REQUIRE(r == CUDA_SUCCESS, CBRS_E_CUDA, "cbrs_dense_tc_bf16: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return CBRS_OK;
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_convert_f32_bf16(const float *x, int64_t ldx, int64_t m, int32_t k, void *out, int64_t ldo, void *stream) {
    CBRS_REQUIRE(x && out, CBRS_E_INVALID, "cbrs_convert_f32_bf16: null pointer");
    CBRS_REQUIRE(m >= 0 && k > 0 && k % 4 == 0 && ldx >= k && ldo >= k && ldx % 4 == 0 && ldo % 4 == 0, CBRS_E_INVALID,
                 "cbrs_convert_f32_bf16: k = %d, ldx = %lld, ldo = %lld (multiples of 4, ld >= k)", k, (long long)ldx, (long long)ldo);
    CBRS_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 7u) == 0, CBRS_E_INVALID,
                 "cbrs_convert_f32_bf16: x must be 16-byte and out 8-byte aligned");
    if (m == 0) return CBRS_OK;
    const int64_t total = m * (int64_t)(k / 4);
    const int blocks = (int)(cdiv(total, 256) < 8 * kSMs ? cdiv(total, 256) : 8 * kSMs);
    convert_f32_bf16_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, m, k, (__nv_bfloat16 *)out, ldo);
    CBRS_CHECK_LAUNCH("cbrs_convert_f32_bf16");
    return CBRS_OK;
}

extern "C" int cbrs_dense_tc_bf16_eligible(int32_t f1, int32_t f2, int32_t n) {
    return f1 > 0 && f1 % kTmKB == 0 && f2 >= 0 && f2 % kTmKB == 0 && n > 0 && n <= 256;
}

extern "C" int cbrs_dense_tc_bf16(const void *x1, int64_t ld1, int64_t rows1, const int64_t *idx1, int32_t f1, const void *x2,
                                  int64_t ld2, int64_t rows2, const int64_t *idx2, int32_t f2, const void *w_image, const float *b,
                                  int64_t m, int32_t n, int act, void *out, int64_t ldo, int out_dtype, void *stream) {
    CBRS_REQUIRE(x1 && w_image && out, CBRS_E_INVALID, "cbrs_dense_tc_bf16: null pointer");
    CBRS_REQUIRE(cbrs_dense_tc_bf16_eligible(f1, f2, n), CBRS_E_INVALID,
                 "cbrs_dense_tc_bf16: f1 = %d, f2 = %d, n = %d (source widths multiples of 64, 1 <= n <= 256)", f1, f2, n);
    CBRS_REQUIRE((f2 == 0) == (x2 == nullptr), CBRS_E_INVALID, "cbrs_dense_tc_bf16: x2 and f2 disagree");
    CBRS_REQUIRE(ld1 >= f1 && ld1 % 8 == 0 && (reinterpret_cast<uintptr_t>(x1) & 15u) == 0 &&
                     (!x2 || (ld2 >= f2 && ld2 % 8 == 0 && (reinterpret_cast<uintptr_t>(x2) & 15u) == 0)),
                 CBRS_E_INVALID, "cbrs_dense_tc_bf16: source rows must be 16-byte aligned (ld %% 8 == 0)");
    CBRS_REQUIRE(rows1 > 0 && rows1 < ((int64_t)1 << 31) && (!x2 || (rows2 > 0 && rows2 < ((int64_t)1 << 31))), CBRS_E_INVALID,
                 "cbrs_dense_tc_bf16: table rows must be in [1, 2^31)");
    CBRS_REQUIRE(m >= 0 && m < ((int64_t)1 << 31), CBRS_E_INVALID, "cbrs_dense_tc_bf16: m out of range");
    CBRS_REQUIRE(idx1 || m <= rows1, CBRS_E_INVALID, "cbrs_dense_tc_bf16: m > rows of x1 without an index");
    CBRS_REQUIRE(!x2 || idx2 || m <= rows2, CBRS_E_INVALID, "cbrs_dense_tc_bf16: m > rows of x2 without an index");
    CBRS_REQUIRE(act >= CBRS_ACT_NONE && act <= CBRS_ACT_TANH, CBRS_E_INVALID, "cbrs_dense_tc_bf16: unknown activation %d", act);
    CBRS_REQUIRE(out_dtype == CBRS_DTYPE_F32 || out_dtype == CBRS_DTYPE_BF16, CBRS_E_INVALID, "cbrs_dense_tc_bf16: out_dtype=%d", out_dtype);
    CBRS_REQUIRE(ldo >= n, CBRS_E_INVALID, "cbrs_dense_tc_bf16: ldo < n");
    CBRS_REQUIRE((reinterpret_cast<uintptr_t>(w_image) & 15u) == 0, CBRS_E_INVALID, "cbrs_dense_tc_bf16: image must be 16-byte aligned");
    if (m == 0) return CBRS_OK;
    TmParams p;
    p.idx1 = idx1; p.idx2 = idx2;
    p.kb1 = f1 / kTmKB; p.kb2 = f2 / kTmKB;
    p.gather1 = idx1 != nullptr; p.gather2 = idx2 != nullptr;
    p.w_image = (const uint8_t *)w_image; p.b = b; p.m = m; p.n = n; p.n_pad = (n + 15) / 16 * 16; p.act = act;
    p.out = out; p.ldo = ldo; p.out_bf16 = out_dtype == CBRS_DTYPE_BF16;
    p.n_tiles = cdiv(m, kTmRows);
    p.stages = tm_stages(p.n_pad);
    p.acc_sets = p.n_pad <= 128 ? 2 : 1;
    CUtensorMap map1, map2;
    int rc = tm_make_map(&map1, x1, ld1, rows1, f1, p.gather1);
    if (rc != CBRS_OK) return rc;
    if (x2) {
        rc = tm_make_map(&map2, x2, ld2, rows2, f2, p.gather2);
        if (rc != CBRS_OK) return rc;
    } else {
        map2 = map1;
    }
    const size_t smem = (size_t)p.stages * (kTmABytes + (size_t)p.n_pad * 128) + tm_tail_bytes(p.n_pad);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(dense_tc_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "cbrs_dense_tc_bf16: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    const unsigned grid = (unsigned)(p.n_tiles < kSMs ? p.n_tiles : kSMs);
    dense_tc_tma_kernel<<<grid, kTmThreads, smem, (cudaStream_t)stream>>>(map1, map2, p);
    CBRS_CHECK_LAUNCH("cbrs_dense_tc_bf16");
    return CBRS_OK;
}
