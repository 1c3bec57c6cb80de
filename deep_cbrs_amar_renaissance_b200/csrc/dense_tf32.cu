// fp32-accurate Dense layer on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), sm_100a: the GCN transform
// Z = X W of /root/reference/src/models/gnn.py:285-295 (spektral GCNConv: transform, then propagate) at config-5 scale.
//
//   out[m, 0:n] = act( X[m, 0:k] @ W[k, n] + b )      X, W, out fp32
//
// The fp32 FFMA kernel (dense.cu) runs this contraction at 34 TFLOP/s: 10.25 ms for the 1.1e7 x 128 x 128 transform of
// config 5, 0.16 of the HBM roofline (profiles/r01_ncu_spmm_dense_v2.csv).  bf16 tensor cores cannot hold the 1e-5
// parity the fp32 path promises, so the product is split ("3xTF32"):  x = xh + xl with xh = tf32(x) (round to nearest,
// 10 mantissa bits) and xl = x - xh (exact in fp32), the same for W, and
//      X W  ~=  Xl Wh + Xh Wl + Xh Wh          (three kind::tf32 MMAs into one fp32 TMEM accumulator)
// The dropped term Xl Wl is below 2^-22 of |x||w| and the tensor core's own truncation of xl / wl to tf32 is of the
// same order, so the result agrees with the fp32 FFMA chain to ~1e-6 of the output scale (tests/test_gpu_tf32.py
// states and checks 1e-5 against the float64 product).
//
// One persistent CTA per SM, 128 output rows per tile, warp-specialised:
//   warp 8    TMA producer: cp.async.bulk.tensor.2d brings the tile's A operand one K atom (32 fp32 = one 128-byte
//             swizzle row) at a time, 128 rows x 128 B (SWIZZLE_128B, so that a thread reading ITS row hits 8 different
//             bank groups), into a ring of landing slots - as many 16 KB slots as fit beside the resident W images
//             (6 at k = n = 128): the bytes in flight per SM are what keeps HBM busy;
//   warps 0-3 split: thread t reads row t of the landed atom into registers, hands the slot straight back to the
//             producer, and writes tf32(x) and x - tf32(x) into TENSOR MEMORY (tcgen05.st, lane = row, column = k;
//             double buffered): the A operand never goes back to shared memory.  v2 of this kernel wrote the two operand
//             tiles to shared memory; with them the kernel moved 160 KB through shared memory per atom (TMA write 16,
//             split read 16 + write 32, MMA reads 12 x (4 + 4)) - 2.8 us per tile at 128 B/clk, as long as the tile's
//             HBM time - now 80 KB;
//   warp 9    one elected thread issues 4 x 3 tcgen05.mma (M=128, N=n, K=8, A from TMEM) per atom and commits: the commit
//             frees the operand buffer; the last commit of a tile hands the accumulator to the epilogue.  Wh and Wl
//             (operand images prepared once per call by cbrs_dense_tf32x3_prepare) stay in shared memory for the CTA's life;
//   warps 4-7 epilogue: tcgen05.ld of the accumulator (double buffered in TMEM when 2 n + 128 <= 512 columns, so tile
//             t+1's MMAs run under tile t's epilogue), bias, activation, 256-bit global stores (a full 32-byte sector per
//             lane), optionally also into the peer-mapped copies of the other GPUs (multi-GPU all-gather from the
//             producing kernel).
// Deep contractions (k >= kT3SplitK): the error of the fp32 accumulator grows linearly with the 3 k / 8 MMAs a tile
// issues into it (measured on a B200: 1.5e-5 of a tile's max |out| at k = 1536, n = 16; 0.56e-5 split).  From
// kT3SplitK on the two cross terms Xl Wh + Xh Wl go to an accumulator of their own, n TMEM columns after the main one,
// which then takes k / 8 MMAs; the epilogue adds the two.  The cross terms are 2^-11 of the product, so their own
// rounding does not count.  Below kT3SplitK the single accumulator stays (and keeps its bits).
// HBM traffic = X once + out once: the kernel's roofline is the copy bandwidth (1.7 ms at config 5).
// Row results do not depend on the row's position in its tile (each accumulator element is an independent dot
// product over K), so a row partition produces the same bits as the full run.
#include "common.cuh"
#include "tc05.cuh"

#include <cuda.h>  // CUtensorMap and its enums; the encoder itself is looked up through the runtime (no -lcuda)

namespace cbrs {

constexpr int kT3Rows = 128;     // output rows per tile = MMA M
constexpr int kT3Atom = 32;      // fp32 elements per 128-byte swizzle row
constexpr int kT3AtomBytes = kT3Rows * 128;   // one operand atom tile: 128 rows x 128 B
constexpr int kT3MaxRaw = 8;     // at most this many landing slots for the TMA loads (16 KB each)
constexpr int kT3Threads = 320;  // 4 split warps, 4 epilogue warps, producer warp, MMA warp
constexpr int kT3SplitK = 384;   // from this k on the cross terms accumulate apart (eligible shapes there have n <= 64)

struct T3Params {
    const uint8_t *w_image;  // [2 (hi, lo)][k_atoms][n][128 B], SWIZZLE_128B, K-major
    const float *bias;
    int32_t act;
    int64_t m;
    int32_t n, k;
    float *out;
    int64_t ldo;
    float *out_peer[CBRS_MAX_PEERS - 1];
    int32_t n_peer;
    int32_t out_bf16;   // out / out_peer hold bf16 (round to nearest even), ldo in elements
    int64_t n_tiles;
    const float *addend; int64_t ld_add;   // optional [m, n] matrix added to the product before bias / row-op (cbrs_dense_tf32x3_ex)
    int32_t l2norm;     // CBRS_ROWOP_L2NORM: v / sqrt(max(sum v^2, 1e-12)) before the activation (GraphSageConv)
    int32_t n_raw;      // landing slots (2 .. kT3MaxRaw)
    int32_t acc_bufs;   // accumulators in TMEM (2 when 2 acc_cols + 128 <= 512 columns, else 1)
    int32_t split_acc;  // k >= kT3SplitK: each accumulator is n main + n cross-term columns (acc_cols = 2 n, else n)
    // GAT row-op (cbrs_dense_tf32x3_attn): p[m] = out[m,:] . a_self, q[m] = out[m,:] . a_neigh (GATConv's attention logits)
    const float *a_self, *a_neigh;
    float *p_out, *q_out;
    float *q_peer[CBRS_MAX_PEERS - 1];
};

__device__ __forceinline__ float t3_act(float v, int act) {
    switch (act) {
        case CBRS_ACT_RELU: return fmaxf(v, 0.f);
        case CBRS_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        case CBRS_ACT_TANH: return tanhf(v);
        default: return v;
    }
}
__device__ __forceinline__ float t3_hi(float x) {   // nearest tf32, low 13 mantissa bits zero
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ void t3_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void t3_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void t3_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
                 : "memory");
}
// 2-D tiled TMA load: box (32 columns, 128 rows) at (col, row); out-of-range rows arrive as zeros
__device__ __forceinline__ void t3_tma_load(void *dst, const CUtensorMap *map, int32_t col, int32_t row, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            tc::smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(col), "r"(row), "r"(tc::smem_u32(bar))
        : "memory");
}
// kind::tf32 instruction descriptor: D fp32, A/B tf32, both K-major, dense
__host__ __device__ constexpr uint32_t t3_idesc(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void t3_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A from tensor memory (lane = row, one 32-bit column per k), B from shared memory
__device__ __forceinline__ void t3_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 32 columns of 32-bit: thread t of the warp writes lane (base_lane + t), columns c..c+31
__device__ __forceinline__ void t3_tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
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
__device__ __forceinline__ void t3_tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void t3_tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 16 fp32 -> 16 bf16 = one 32-byte sector
__device__ __forceinline__ void t3_store16_bf16(float *base, int64_t elem, const float (&o)[2][8]) {
    uint32_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = tc::pack_bf16x2(o[j >> 2][(2 * j) & 7], o[j >> 2][(2 * j + 1) & 7]);
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(reinterpret_cast<__nv_bfloat16 *>(base) + elem),
                 "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                 : "memory");
}
__device__ __forceinline__ void t3_store8(float *p, const float (&o)[8]) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]),
                 "f"(o[4]), "f"(o[5]), "f"(o[6]), "f"(o[7])
                 : "memory");
}

// W [k, n] fp32 (Keras [in, out]) -> two B operand images (hi = tf32(W), lo = W - hi): element (col, kk) of atom a at
// a*n*128 + sw128(col, kk/4) + (kk%4)*4, K-major.  lo image follows the hi image.
__global__ void t3_prep_kernel(const float *__restrict__ w, int k, int n, uint8_t *__restrict__ image) {
    const int64_t total = (int64_t)k * n;
    const int64_t img = (int64_t)(k / kT3Atom) * n * 128;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int kg = (int)(e / n), col = (int)(e % n);
        const float v = w[e];
        const float hi = t3_hi(v);
        const int a = kg / kT3Atom, kk = kg % kT3Atom;
        const size_t off = (size_t)a * n * 128 + tc::sw128_offset(col, kk >> 2) + (kk & 3) * 4;
        *reinterpret_cast<float *>(image + off) = hi;
        *reinterpret_cast<float *>(image + img + off) = v - hi;
    }
}

// kPlain: no bias, no activation (the GCN / GAT transform): the epilogue is a straight copy.  kAttn (implies kPlain):
// also the two attention logits of the row.
template <bool kPlain, bool kAttn = false>
__global__ void __launch_bounds__(kT3Threads, 1)
    dense_tf32x3_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ T3Params p) {
    extern __shared__ __align__(1024) unsigned char t3_smem[];
    const int k_atoms = p.k / kT3Atom;
    const int w_bytes = k_atoms * p.n * 128;           // one image (hi or lo)
    unsigned char *Wh = t3_smem;                       // [k_atoms][n][128 B]
    unsigned char *Wl = Wh + w_bytes;
    unsigned char *raw_s = Wl + w_bytes;               // [n_raw][16 KB]: where TMA lands the fp32 atoms
    uint64_t *bars = reinterpret_cast<uint64_t *>(raw_s + (size_t)p.n_raw * kT3AtomBytes);
    uint64_t *raw_full = bars, *raw_empty = bars + kT3MaxRaw, *op_ready = bars + 2 * kT3MaxRaw, *op_empty = op_ready + 2;
    uint64_t *acc_full = op_empty + 2, *acc_empty = acc_full + 2, *w_full = acc_empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(w_full + 1);
    float *bias_s = reinterpret_cast<float *>(tmem_slot + 2);
    // TMEM columns: accumulators [0, acc_bufs acc_cols) (each: n main columns, then n cross-term columns when split),
    // then the split operand, double buffered: (hi 32 | lo 32) x 2
    const uint32_t acc_cols = (uint32_t)(p.n << p.split_acc);
    const uint32_t col_a = (uint32_t)p.acc_bufs * acc_cols;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint32_t tmem_cols = 32;
    while (tmem_cols < col_a + 128) tmem_cols <<= 1;
    if ((tc::smem_u32(t3_smem) & 1023u) != 0u) __trap();  // SWIZZLE_128B tiles need the declared alignment

    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 32) {
        for (int s = 0; s < p.n_raw; ++s) {
            tc::mbar_init(raw_full + s, 1);
            tc::mbar_init(raw_empty + s, 128);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(op_ready + a, 128);
            tc::mbar_init(op_empty + a, 1);
            tc::mbar_init(acc_full + a, 1);
            tc::mbar_init(acc_empty + a, 128);
        }
        tc::mbar_init(w_full, 1);
        tc::fence_mbar_init();
    }
    if (!kPlain)
        for (int e = tid; e < p.n; e += kT3Threads) bias_s[e] = p.bias ? __ldg(p.bias + e) : 0.f;
    if (kAttn)
        for (int e = tid; e < p.n; e += kT3Threads) {
            bias_s[e] = __ldg(p.a_self + e);
            bias_s[p.n + e] = __ldg(p.a_neigh + e);
        }
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t zero_rt = (uint32_t)p.n >> 20;   // 0 (n <= 256), but not to the compiler
    const int64_t my_tiles = (p.n_tiles > (int64_t)blockIdx.x) ? (p.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp == 8) {
        // ---------------- TMA producer ----------------
        if (tc::elect_one()) {   // one lane, and ptxas knows it: TMA / MMA instructions issue once, not in a per-lane loop
            t3_expect_tx(w_full, 2u * (uint32_t)w_bytes);
            for (int off = 0; off < 2 * w_bytes; off += 16384) {
                const int nb = (2 * w_bytes - off < 16384) ? 2 * w_bytes - off : 16384;
                t3_bulk_g2s(Wh + off, p.w_image + off, (uint32_t)nb, w_full);
            }
            int64_t it = 0;
            for (int64_t lt = 0; lt < my_tiles; ++lt) {
                const int64_t tile = blockIdx.x + lt * gridDim.x;
                for (int a = 0; a < k_atoms; ++a, ++it) {
                    const int s = (int)(it % p.n_raw);
                    const int64_t use = it / p.n_raw;
                    if (use > 0) tc::mbar_wait(raw_empty + s, (uint32_t)(use - 1) & 1u);
                    t3_expect_tx(raw_full + s, kT3AtomBytes);
                    t3_tma_load(raw_s + s * kT3AtomBytes, &map_x, a * kT3Atom, (int32_t)(tile * kT3Rows), raw_full + s);
                }
            }
        }
    } else if (warp == 9) {
        // ---------------- MMA issuer ----------------
        if (tc::elect_one()) {
            const uint32_t idesc = t3_idesc(kT3Rows, p.n);
            const uint32_t wh_addr = tc::smem_u32(Wh), wl_addr = tc::smem_u32(Wl);
            tc::mbar_wait(w_full, 0);
            int64_t it = 0;
            for (int64_t lt = 0; lt < my_tiles; ++lt) {
                const int acc = (int)(lt % p.acc_bufs);
                const int64_t acc_use = lt / p.acc_bufs;
                if (acc_use > 0) tc::mbar_wait(acc_empty + acc, (uint32_t)(acc_use - 1) & 1u);
                tc::tc_fence_after_sync();
                const uint32_t d = tmem_base + (uint32_t)acc * acc_cols;
                const uint32_t dx = p.split_acc ? d + (uint32_t)p.n : d;   // where the cross terms accumulate
                for (int a = 0; a < k_atoms; ++a, ++it) {
                    const int o = (int)(it & 1);
                    tc::mbar_wait(op_ready + o, (uint32_t)(it >> 1) & 1u);
                    tc::tc_fence_after_sync();
                    const uint32_t ah = tmem_base + col_a + (uint32_t)o * 64, al = ah + 32;
                    const uint32_t bh = wh_addr + (uint32_t)a * p.n * 128, bl = wl_addr + (uint32_t)a * p.n * 128;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {   // 4 x K=8 inside the 32-wide atom; small terms first
                        const uint32_t koff = (uint32_t)ks * 32;
                        const uint32_t more = (a > 0 || ks > 0) ? 1u : 0u;
                        t3_mma_ts(dx, al + (uint32_t)ks * 8, tc::smem_desc_sw128(bh + koff), idesc, more);
                        t3_mma_ts(dx, ah + (uint32_t)ks * 8, tc::smem_desc_sw128(bl + koff), idesc, 1u);
                        t3_mma_ts(d, ah + (uint32_t)ks * 8, tc::smem_desc_sw128(bh + koff), idesc, p.split_acc ? more : 1u);
                    }
                    tc::mma_commit(op_empty + o);       // operand buffer reusable once these MMAs have read it
                }
                tc::mma_commit(acc_full + acc);         // accumulator complete
            }
        }
    } else if (warp < 4) {
        // ---------------- split: x -> (tf32(x), x - tf32(x)), thread t = row t of the tile ----------------
        // The landing slot is given back to the producer as soon as the thread's row sits in registers, so a slot is
        // held for one HBM round trip only; the split operand goes straight into tensor memory.
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + col_a;
        int64_t it = 0;
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            for (int a = 0; a < k_atoms; ++a, ++it) {
                const int s = (int)(it % p.n_raw), o = (int)(it & 1);
                tc::mbar_wait(raw_full + s, (uint32_t)(it / p.n_raw) & 1u);
                const unsigned char *raw = raw_s + s * kT3AtomBytes + tid * 128;   // my row; chunk c sits at c ^ (row & 7)
                float4 v[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) v[c] = *reinterpret_cast<const float4 *>(raw + ((c ^ (tid & 7)) << 4));
                // the slot may be refilled only after every load of it has RETURNED: the barrier address carries a data
                // dependence on all 32 loaded words (a run-time zero the compiler cannot fold), so the arrive cannot
                // issue - let alone be reordered by ptxas - before the loads have landed in registers
                uint32_t dep = 0u;
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    dep ^= __float_as_uint(v[c].x) ^ __float_as_uint(v[c].y) ^ __float_as_uint(v[c].z) ^ __float_as_uint(v[c].w);
                t3_arrive(reinterpret_cast<uint64_t *>(reinterpret_cast<unsigned char *>(raw_empty + s) + (dep & zero_rt)));
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float h0 = t3_hi(v[c].x), h1 = t3_hi(v[c].y), h2 = t3_hi(v[c].z), h3 = t3_hi(v[c].w);
                    hi[4 * c] = __float_as_uint(h0); hi[4 * c + 1] = __float_as_uint(h1);
                    hi[4 * c + 2] = __float_as_uint(h2); hi[4 * c + 3] = __float_as_uint(h3);
                    lo[4 * c] = __float_as_uint(v[c].x - h0); lo[4 * c + 1] = __float_as_uint(v[c].y - h1);
                    lo[4 * c + 2] = __float_as_uint(v[c].z - h2); lo[4 * c + 3] = __float_as_uint(v[c].w - h3);
                }
                if (it >= 2) {   // the MMAs that read this operand buffer two atoms ago must have completed
                    tc::mbar_wait(op_empty + o, (uint32_t)((it >> 1) - 1) & 1u);
                    tc::tc_fence_after_sync();
                }
                t3_tmem_st32(trow + (uint32_t)o * 64, hi);
                t3_tmem_st32(trow + (uint32_t)o * 64 + 32, lo);
                t3_tmem_st_wait();
                tc::tc_fence_before_sync();     // my tcgen05.st -> ordered before the MMAs the issuer launches after the arrive
                t3_arrive(op_ready + o);
            }
        }
    } else {
        // ---------------- epilogue (warps 4..7: TMEM lane quadrant = warp & 3) ----------------
        const int quad = warp & 3;
        const bool v8_ok = (p.ldo % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 31u) == 0);
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            const int64_t tile = blockIdx.x + lt * gridDim.x;
            const int acc = (int)(lt % p.acc_bufs);
            tc::mbar_wait(acc_full + acc, (uint32_t)(lt / p.acc_bufs) & 1u);
            tc::tc_fence_after_sync();
            const int64_t row = tile * kT3Rows + quad * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)acc * acc_cols;
            // columns cb..cb+15 of the accumulator (warp-collective); cross: add the split-off cross terms
            auto ld_acc = [&](int cb, uint32_t (&v)[16], bool cross) {
                tc::tmem_ld16(taddr + (uint32_t)cb, v);
                if (cross) {
                    uint32_t c[16];
                    tc::tmem_ld16(taddr + (uint32_t)(p.n + cb), c);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(c[j]));
                } else {
                    tc::tmem_ld_wait();
                }
            };
            float ps = 0.f, qs = 0.f;
            float scale = 1.f;
            const float *arow = (!kPlain && p.addend && row < p.m) ? p.addend + row * p.ld_add : nullptr;
            bool folded = false;   // the accumulator already holds product + addend + bias (first pass of the row-op)
            if (!kPlain && (p.l2norm || p.addend)) {
                // first pass over the accumulator: x = product + addend + bias, written back into the accumulator's own
                // TMEM columns (the addend is read from HBM once: 64 contiguous bytes per lane and block, the next
                // block's four 128-bit loads in flight while this one is processed), and the row's sum of squares
                float ss = 0.f;
                float4 a_cur[4], a_nxt[4];
                auto load_add = [&](int cb, float4 (&a)[4]) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) a[q] = arow ? ldg4(arow + cb + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                };
                load_add(0, a_cur);
                for (int cb = 0; cb < p.n; cb += 16) {
                    if (cb + 16 < p.n) load_add(cb + 16, a_nxt);
                    uint32_t v[16];
                    ld_acc(cb, v, p.split_acc);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 bb = *reinterpret_cast<const float4 *>(bias_s + cb + 4 * q);
                        const float x0 = __uint_as_float(v[4 * q]) + a_cur[q].x + bb.x, x1 = __uint_as_float(v[4 * q + 1]) + a_cur[q].y + bb.y;
                        const float x2 = __uint_as_float(v[4 * q + 2]) + a_cur[q].z + bb.z, x3 = __uint_as_float(v[4 * q + 3]) + a_cur[q].w + bb.w;
                        ss = fmaf(x0, x0, ss); ss = fmaf(x1, x1, ss); ss = fmaf(x2, x2, ss); ss = fmaf(x3, x3, ss);
                        v[4 * q] = __float_as_uint(x0); v[4 * q + 1] = __float_as_uint(x1);
                        v[4 * q + 2] = __float_as_uint(x2); v[4 * q + 3] = __float_as_uint(x3);
                    }
                    t3_tmem_st16(taddr + (uint32_t)cb, v);
#pragma unroll
                    for (int q = 0; q < 4; ++q) a_cur[q] = a_nxt[q];
                }
                t3_tmem_st_wait();
                if (p.l2norm) scale = 1.f / sqrtf(fmaxf(ss, 1e-12f));
                folded = true;
            }
            for (int cb = 0; cb < p.n; cb += 16) {
                uint32_t v[16];
                ld_acc(cb, v, p.split_acc && !folded);   // a folded accumulator already holds the cross terms
                if (row < p.m) {
                    float o[2][8];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        if (kPlain) {
                            o[j >> 3][j & 7] = __uint_as_float(v[j]);
                        } else {
                            const float x = folded ? __uint_as_float(v[j]) : __uint_as_float(v[j]) + bias_s[cb + j];
                            o[j >> 3][j & 7] = t3_act(x * scale, p.act);
                        }
                    }
                    if (kAttn) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            ps = fmaf(o[j >> 3][j & 7], bias_s[cb + j], ps);
                            qs = fmaf(o[j >> 3][j & 7], bias_s[p.n + cb + j], qs);
                        }
                    }
                    const int64_t off = row * p.ldo + cb;
                    if (p.out_bf16) {   // host checked: ldo % 16 == 0 and 32-byte aligned bases
                        t3_store16_bf16(p.out, off, o);
                        for (int q = 0; q < p.n_peer; ++q) t3_store16_bf16(p.out_peer[q], off, o);
                    } else if (v8_ok) {
                        t3_store8(p.out + off, o[0]);
                        t3_store8(p.out + off + 8, o[1]);
                        for (int q = 0; q < p.n_peer; ++q) {
                            t3_store8(p.out_peer[q] + off, o[0]);
                            t3_store8(p.out_peer[q] + off + 8, o[1]);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) p.out[off + j] = o[j >> 3][j & 7];
                        for (int q = 0; q < p.n_peer; ++q)
#pragma unroll
                            for (int j = 0; j < 16; ++j) p.out_peer[q][off + j] = o[j >> 3][j & 7];
                    }
                }
            }
            if (kAttn && row < p.m) {
                p.p_out[row] = ps;
                p.q_out[row] = qs;
                for (int q = 0; q < p.n_peer; ++q) p.q_peer[q][row] = qs;
            }
            tc::tc_fence_before_sync();
            t3_arrive(acc_empty + acc);
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, tmem_cols);
    }
}

static size_t t3_tail_bytes(int n) { return (2 * kT3MaxRaw + 9) * sizeof(uint64_t) + 8 + 2 * (size_t)n * 4 + 64; }
// landing slots that fit beside the resident W images (0: the shape does not fit at all)
static int t3_raw_slots(int k, int n) {
    const size_t fixed = 2 * (size_t)(k / kT3Atom) * n * 128 + t3_tail_bytes(n);
    if (fixed + 2 * (size_t)kT3AtomBytes > 227 * 1024) return 0;
    const size_t slots = (227 * 1024 - fixed) / kT3AtomBytes;
    return slots > (size_t)kT3MaxRaw ? kT3MaxRaw : (int)slots;
}
static size_t t3_smem_bytes(int k, int n) {
    return 2 * (size_t)(k / kT3Atom) * n * 128 + (size_t)t3_raw_slots(k, n) * kT3AtomBytes + t3_tail_bytes(n);
}

typedef CUresult (*t3_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                 const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static t3_encode_fn t3_encoder() {
    static t3_encode_fn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (t3_encode_fn)ptr;
    }
    return fn;
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_dense_tf32x3_eligible(int32_t k, int32_t n) {
    return k > 0 && k % kT3Atom == 0 && n >= 16 && n <= 256 && n % 16 == 0 && t3_raw_slots(k, n) >= 2;
}

extern "C" size_t cbrs_dense_tf32x3_image_bytes(int32_t k, int32_t n) {
    if (!cbrs_dense_tf32x3_eligible(k, n)) return 0;
    return 2 * (size_t)(k / kT3Atom) * n * 128;
}

extern "C" int cbrs_dense_tf32x3_prepare(const float *w, int32_t k, int32_t n, void *image, void *stream) {
    CBRS_REQUIRE(w && image, CBRS_E_INVALID, "cbrs_dense_tf32x3_prepare: null pointer");
    CBRS_REQUIRE(cbrs_dense_tf32x3_eligible(k, n), CBRS_E_INVALID,
                 "cbrs_dense_tf32x3_prepare: k = %d, n = %d (k %% 32 == 0, n %% 16 == 0, 16 <= n <= 256, operands must fit "
                 "shared memory)", k, n);
    CBRS_REQUIRE((reinterpret_cast<uintptr_t>(image) & 15u) == 0, CBRS_E_INVALID, "cbrs_dense_tf32x3_prepare: image must be 16-byte aligned");
    const int64_t total = (int64_t)k * n;
    const int blocks = (int)(cdiv(total, 256) < 4 * kSMs ? cdiv(total, 256) : 4 * kSMs);
    t3_prep_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, k, n, (uint8_t *)image);
    CBRS_CHECK_LAUNCH("cbrs_dense_tf32x3_prepare");
    return CBRS_OK;
}

static int t3_impl(const float *x, int64_t ldx, const void *w_image, const float *b, const float *addend, int64_t ld_add, int rowop,
                   int64_t m, int32_t k, int32_t n, int act,
                   void *out_v, int64_t ldo, int out_dtype, void *const *out_peers_host, int n_peers, const float *a_self,
                   const float *a_neigh, float *p_out, float *q_out, void *const *q_peers_host, void *stream) {
    float *out = (float *)out_v;
    const bool attn = a_self != nullptr;
    CBRS_REQUIRE(!attn || (a_neigh && p_out && q_out && !b && act == CBRS_ACT_NONE && out_dtype == CBRS_DTYPE_F32 &&
                           (n_peers == 0 || q_peers_host)),
                 CBRS_E_INVALID, "cbrs_dense_tf32x3_attn: needs a_self, a_neigh, p_out, q_out (and q_peers with peers), fp32 output");
    CBRS_REQUIRE(out_dtype == CBRS_DTYPE_F32 || out_dtype == CBRS_DTYPE_BF16, CBRS_E_INVALID, "cbrs_dense_tf32x3: out_dtype=%d", out_dtype);
    CBRS_REQUIRE(out_dtype == CBRS_DTYPE_F32 || (ldo % 16 == 0 && (reinterpret_cast<uintptr_t>(out_v) & 31u) == 0), CBRS_E_INVALID,
                 "cbrs_dense_tf32x3: a bf16 output needs 32-byte aligned rows (ldo %% 16 == 0)");
    CBRS_REQUIRE(x && w_image && out, CBRS_E_INVALID, "cbrs_dense_tf32x3: null pointer");
    CBRS_REQUIRE(rowop == CBRS_ROWOP_NONE || rowop == CBRS_ROWOP_L2NORM, CBRS_E_INVALID, "cbrs_dense_tf32x3: rowop %d (none or l2norm)", rowop);
    CBRS_REQUIRE(!attn || (!addend && rowop == CBRS_ROWOP_NONE), CBRS_E_INVALID, "cbrs_dense_tf32x3_attn takes no addend / row-op");
    CBRS_REQUIRE(!addend || (ld_add >= n && ld_add % 4 == 0 && (reinterpret_cast<uintptr_t>(addend) & 15u) == 0), CBRS_E_INVALID,
                 "cbrs_dense_tf32x3: addend rows must be 16-byte aligned (ld_add %% 4 == 0, ld_add >= n)");
    CBRS_REQUIRE(cbrs_dense_tf32x3_eligible(k, n), CBRS_E_INVALID, "cbrs_dense_tf32x3: k = %d, n = %d not supported (see "
                 "cbrs_dense_tf32x3_eligible); use cbrs_dense", k, n);
    CBRS_REQUIRE(m >= 0 && m < ((int64_t)1 << 31) && ldx >= k && ldo >= n, CBRS_E_INVALID, "cbrs_dense_tf32x3: bad shape");
    CBRS_REQUIRE(ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0, CBRS_E_INVALID,
                 "cbrs_dense_tf32x3: rows of x must be 16-byte aligned (TMA global stride)");
    CBRS_REQUIRE((reinterpret_cast<uintptr_t>(w_image) & 15u) == 0, CBRS_E_INVALID, "cbrs_dense_tf32x3: image must be 16-byte aligned");
    CBRS_REQUIRE(act >= CBRS_ACT_NONE && act <= CBRS_ACT_TANH, CBRS_E_INVALID, "cbrs_dense_tf32x3: unknown activation %d", act);
    CBRS_REQUIRE(n_peers >= 0 && n_peers < CBRS_MAX_PEERS && (n_peers == 0 || out_peers_host), CBRS_E_INVALID,
                 "cbrs_dense_tf32x3: n_peers=%d", n_peers);
    if (m == 0) return CBRS_OK;
    t3_encode_fn encode = t3_encoder();
    CBRS_REQUIRE(encode, CBRS_E_CUDA, "cbrs_dense_tf32x3: cuTensorMapEncodeTiled is not available from this driver");
    CUtensorMap map;
    const cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)m};
    const cuuint64_t strides[1] = {(cuuint64_t)ldx * 4};
    const cuuint32_t box[2] = {(cuuint32_t)kT3Atom, (cuuint32_t)kT3Rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(x), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CBRS_REQUIRE(r == CUDA_SUCCESS, CBRS_E_CUDA, "cbrs_dense_tf32x3: cuTensorMapEncodeTiled failed (%d)", (int)r);
    T3Params p;
    p.w_image = (const uint8_t *)w_image; p.bias = b; p.act = act; p.m = m; p.n = n; p.k = k; p.out = out; p.ldo = ldo;
    p.n_peer = n_peers;
    p.out_bf16 = out_dtype == CBRS_DTYPE_BF16;
    for (int q = 0; q < CBRS_MAX_PEERS - 1; ++q) {
        p.out_peer[q] = q < n_peers ? (float *)out_peers_host[q] : nullptr;
        CBRS_REQUIRE(q >= n_peers || (p.out_peer[q] && ((reinterpret_cast<uintptr_t>(p.out_peer[q]) & 31u) ==
                                                         (reinterpret_cast<uintptr_t>(out) & 31u))),
                     CBRS_E_INVALID, "cbrs_dense_tf32x3: peer copy %d is null or aligned differently from out", q);
    }
    p.a_self = a_self; p.a_neigh = a_neigh; p.p_out = p_out; p.q_out = q_out;
    for (int q = 0; q < CBRS_MAX_PEERS - 1; ++q) {
        p.q_peer[q] = (attn && q < n_peers) ? (float *)q_peers_host[q] : nullptr;
        CBRS_REQUIRE(!attn || q >= n_peers || p.q_peer[q], CBRS_E_INVALID, "cbrs_dense_tf32x3_attn: q peer copy %d is null", q);
    }
    p.addend = addend; p.ld_add = ld_add; p.l2norm = rowop == CBRS_ROWOP_L2NORM;
    p.n_tiles = cdiv(m, kT3Rows);
    p.n_raw = t3_raw_slots(k, n);
    p.split_acc = k >= kT3SplitK ? 1 : 0;
    p.acc_bufs = (2 * (n << p.split_acc) + 128 <= 512) ? 2 : 1;
    const size_t smem = t3_smem_bytes(k, n);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(dense_tf32x3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(dense_tf32x3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(dense_tf32x3_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "cbrs_dense_tf32x3: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    const unsigned grid = (unsigned)(p.n_tiles < kSMs ? p.n_tiles : kSMs);
    if (attn)
        dense_tf32x3_kernel<true, true><<<grid, kT3Threads, smem, (cudaStream_t)stream>>>(map, p);
    else if (!b && act == CBRS_ACT_NONE && !addend && rowop == CBRS_ROWOP_NONE)
        dense_tf32x3_kernel<true><<<grid, kT3Threads, smem, (cudaStream_t)stream>>>(map, p);
    else
        dense_tf32x3_kernel<false><<<grid, kT3Threads, smem, (cudaStream_t)stream>>>(map, p);
    CBRS_CHECK_LAUNCH("cbrs_dense_tf32x3");
    return CBRS_OK;
}

extern "C" int cbrs_dense_tf32x3(const float *x, int64_t ldx, const void *w_image, const float *b, int64_t m, int32_t k,
                                 int32_t n, int act, void *out, int64_t ldo, int out_dtype, void *const *out_peers_host,
                                 int n_peers, void *stream) {
    return t3_impl(x, ldx, w_image, b, nullptr, 0, CBRS_ROWOP_NONE, m, k, n, act, out, ldo, out_dtype, out_peers_host, n_peers, nullptr,
                   nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int cbrs_dense_tf32x3_ex(const float *x, int64_t ldx, const void *w_image, const float *b, const float *addend,
                                    int64_t ld_add, int rowop, int64_t m, int32_t k, int32_t n, int act, void *out, int64_t ldo,
                                    int out_dtype, void *const *out_peers_host, int n_peers, void *stream) {
    return t3_impl(x, ldx, w_image, b, addend, ld_add, rowop, m, k, n, act, out, ldo, out_dtype, out_peers_host, n_peers, nullptr,
                   nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int cbrs_dense_tf32x3_attn(const float *x, int64_t ldx, const void *w_image, int64_t m, int32_t k, int32_t n,
                                      const float *a_self, const float *a_neigh, float *p_out, float *q_out, float *out,
                                      int64_t ldo, void *const *out_peers_host, void *const *q_peers_host, int n_peers,
                                      void *stream) {
    CBRS_REQUIRE(a_self && a_neigh && p_out && q_out, CBRS_E_INVALID, "cbrs_dense_tf32x3_attn: null attention argument");
    return t3_impl(x, ldx, w_image, nullptr, nullptr, 0, CBRS_ROWOP_NONE, m, k, n, CBRS_ACT_NONE, out, ldo, CBRS_DTYPE_F32, out_peers_host, n_peers, a_self,
                   a_neigh, p_out, q_out, q_peers_host, stream);
}
