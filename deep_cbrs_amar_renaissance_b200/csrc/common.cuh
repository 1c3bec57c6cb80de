// Internal helpers shared by the sm_100a kernels.  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/cbrs_b200.h"

namespace cbrs {

void set_error(const char *fmt, ...);

#define CBRS_REQUIRE(cond, code, ...)            \
    do {                                         \
        if (!(cond)) {                           \
            ::cbrs::set_error(__VA_ARGS__);      \
            return (code);                       \
        }                                        \
    } while (0)

// launch check: catches configuration errors without synchronising
#define CBRS_CHECK_LAUNCH(what)                                                         \
    do {                                                                                \
        cudaError_t e__ = cudaGetLastError();                                           \
        if (e__ != cudaSuccess) {                                                       \
            ::cbrs::set_error("%s: %s", (what), cudaGetErrorString(e__));               \
            return CBRS_E_CUDA;                                                         \
        }                                                                               \
    } while (0)

constexpr int kSMs = 148;  // B200: 2 dies x 74 SMs

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// bump allocator over the caller's workspace
struct Arena {
    char *base;
    size_t cap, off;
    Arena(void *p, size_t n) : base((char *)p), cap(n), off(0) {}
    template <typename T>
    T *take(size_t count) {
        size_t bytes = align_up(count * sizeof(T));
        if (off + bytes > cap) return nullptr;
        T *r = (T *)(base + off);
        off += bytes;
        return r;
    }
};

// ---- scan / sort primitives (scan_sort.cu) --------------------------------
size_t scan_u32_workspace_bytes(int64_t n);
// in-place exclusive scan; *total_out (device uint32, may be null) receives the sum
int scan_u32_exclusive(uint32_t *data, int64_t n, uint32_t *total_out, void *ws, size_t ws_bytes,
                       cudaStream_t s);
size_t scan_i64_workspace_bytes(int64_t n);
int scan_i64_exclusive(int64_t *data, int64_t n, int64_t *total_out, void *ws, size_t ws_bytes,
                       cudaStream_t s);
size_t sort_workspace_bytes(int64_t n);
// stable LSD radix sort; result is left in keys/payload (copied back if needed)
int sort_pairs_u64(uint64_t *keys, uint32_t *payload, int64_t n, int key_bits, void *ws,
                   size_t ws_bytes, cudaStream_t s);

// ---- device helpers ---------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

// streaming (read-once) loads: keep them out of L1 so gathered rows stay cached
__device__ __forceinline__ int ld_stream_i32(const int32_t *p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// Catalog exclusion lists (CSR; contract in include/cbrs_b200.h): is `item` in row `row`'s list?  A lower-bound binary
// search over [rowptr[row], rowptr[row + 1]): at most log2(len) + 1 probes, never a read outside that range, so an
// unsorted row can only miss some of its own items.  Null lists exclude nothing.  The fused scorers call it only for
// a candidate that beats the user's current k-th key, so the search runs rarely; they are instantiated twice
// (template flag kExcl) so that a call without lists runs the kernel without the check at all.
__device__ __forceinline__ bool excluded_item(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ items,
                                              int64_t row, int32_t item) {
    if (rowptr == nullptr) return false;
    int64_t lo = __ldg(rowptr + row);
    const int64_t end = __ldg(rowptr + row + 1);
    int64_t hi = end;
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(items + mid) < item) lo = mid + 1; else hi = mid;
    }
    return lo < end && __ldg(items + lo) == item;
}

// Candidate lists of the tensor-core catalog scorers (score_tf32.cu, score_hybrid_tf32.cu): 64-bit keys
// (orderable(logit) << 32) | ~item, so that a larger key is a higher score, ties going to the lower item id.
__device__ __forceinline__ uint32_t orderable_f32(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float from_orderable_f32(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
// one warp: keep the best min(k, n) keys of c[0..n) in c[0..), descending; *thr becomes the k-th key once k are held
static __device__ void topk_compact(unsigned long long *c, int *cnt, unsigned long long *thr, int k, int lane) {
    const int n = *cnt;
    const int keep = n < k ? n : k;
    for (int r = 0; r < keep; ++r) {
        unsigned long long best = 0ull;
        int bi = -1;
        for (int i = r + lane; i < n; i += 32) {
            const unsigned long long v = c[i];
            if (v > best) { best = v; bi = i; }
        }
        unsigned long long m = best;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
            m = t > m ? t : m;
        }
        if (best == m && bi >= 0) {
            c[bi] = c[r];
            c[r] = m;
        }
        __syncwarp();
    }
    if (lane == 0) {
        *cnt = keep;
        *thr = (keep == k) ? c[k - 1] : 0ull;
    }
    __syncwarp();
}

}  // namespace cbrs
