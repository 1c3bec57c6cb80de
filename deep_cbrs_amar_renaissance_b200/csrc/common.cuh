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

// ---- per-user candidate lists of the fused catalog scorers (score*.cu) --------------------------------------------
// A CTA keeps, for each of its users, a list of 64-bit keys (orderable(value) << 32) | ~item in shared memory: a larger
// key is a higher value, ties going to the lower item id, so the result does not depend on insertion order.  Key 0 is
// below every real key (the low word of one is ~item >= 2^31).  A candidate is appended (topk_offer) when it beats the
// user's current k-th key; before every item tile a list that could overflow is cut back to its best k
// (topk_make_room), and at the end topk_write compacts once more and writes the k slots.  The loop over users, and
// which warp owns user ul, stay with each kernel: a list is only ever touched by one warp at a time.

// order-preserving map float -> uint32 (ascending)
__device__ __forceinline__ uint32_t orderable_f32(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float from_orderable_f32(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ unsigned long long topk_key(float value, uint32_t item) {
    return ((unsigned long long)orderable_f32(value) << 32) | (unsigned long long)(0xffffffffu - item);
}
__device__ __forceinline__ int32_t topk_key_item(unsigned long long key) {
    return (int32_t)(0xffffffffu - (uint32_t)(key & 0xffffffffull));
}
__device__ __forceinline__ float topk_key_value(unsigned long long key) { return from_orderable_f32((uint32_t)(key >> 32)); }

// one output slot: the item and value of `key` (kSigmoid: the value is a logit, written as its sigmoid), or (-1, -inf)
// for key 0, a slot the list has no item for
template <bool kSigmoid>
__device__ __forceinline__ void topk_store(unsigned long long key, int32_t *id, float *score) {
    if (key != 0ull) {
        *id = topk_key_item(key);
        const float v = topk_key_value(key);
        *score = kSigmoid ? 1.f / (1.f + expf(-v)) : v;
    } else {
        *id = -1;
        *score = -INFINITY;
    }
}

constexpr int kTopkTile = 32;   // most candidates one item tile adds to a user's list
// a compaction keeps k keys, so a list of 2k + 32 takes one more tile whenever it holds at most 2k
__host__ __device__ constexpr int topk_list_cap(int k) { return 2 * k + kTopkTile; }
// shared memory of tu lists: keys [tu][cap], k-th keys [tu] (0 until k are held), counts [tu]
static inline size_t topk_lists_smem_bytes(int tu, int k) {
    return (size_t)tu * topk_list_cap(k) * 8 + (size_t)tu * 8 + (size_t)tu * 4;
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

// The three operations below address the lists of a CTA's users as in shared memory: keys cand [tu][cap] with
// cap = topk_list_cap(k), k-th keys thr [tu], counts cnt [tu]; ul is the user's slot in the CTA.

// one warp, before an item tile: compact user ul's list if it might not have room for the tile's candidates
__device__ __forceinline__ void topk_make_room(unsigned long long *cand, int *cnt, unsigned long long *thr, int cap, int ul,
                                               int k, int lane) {
    if (cnt[ul] > cap - kTopkTile) topk_compact(cand + ul * cap, cnt + ul, thr + ul, k, lane);
}

// one thread: append (value, item) to user ul's list if it beats the list's k-th key and is not on the exclusion list of
// `user`, the user's global row (kExcl)
template <bool kExcl>
__device__ __forceinline__ void topk_offer(unsigned long long *cand, int *cnt, const unsigned long long *thr, int cap, int ul,
                                           float value, int32_t item, int64_t user, const int64_t *__restrict__ excl_rowptr,
                                           const int32_t *__restrict__ excl_items) {
    const unsigned long long key = topk_key(value, (uint32_t)item);
    if (key > thr[ul] && !(kExcl && excluded_item(excl_rowptr, excl_items, user, item))) {
        const int pos = atomicAdd(cnt + ul, 1);
        cand[ul * cap + pos] = key;   // pos < cap: topk_make_room ran before this tile
    }
}

// one warp, after the last tile: user ul's k slots to rows user * k .. user * k + k - 1 of ids_out / scores_out (nothing
// for a user at or past n_users, the CTA's padding); kSigmoid as in topk_store
template <bool kSigmoid>
__device__ __forceinline__ void topk_write(unsigned long long *cand, int *cnt, unsigned long long *thr, int cap, int ul,
                                           int k, int lane, int64_t user, int64_t n_users, int32_t *ids_out,
                                           float *scores_out) {
    unsigned long long *c = cand + ul * cap;
    topk_compact(c, cnt + ul, thr + ul, k, lane);
    if (user >= n_users) return;
    const int n = cnt[ul];
    for (int r = lane; r < k; r += 32) {
        const int64_t o = user * k + r;
        topk_store<kSigmoid>(r < n ? c[r] : 0ull, ids_out + o, scores_out + o);
    }
}

// ---- host side of the fused catalog scorers -------------------------------------------------------------------------
// the argument rules they all share; `who` prefixes the messages
static inline int check_catalog_args(const char *who, const int64_t *excl_rowptr, const int32_t *excl_items,
                                     int64_t n_users, int32_t n_items, int32_t k) {
    CBRS_REQUIRE(!excl_rowptr == !excl_items, CBRS_E_INVALID, "%s: %s is null but %s is not", who,
                 excl_rowptr ? "excl_items" : "excl_rowptr", excl_rowptr ? "excl_rowptr" : "excl_items");
    CBRS_REQUIRE(n_users >= 0 && n_items > 0 && k > 0 && k <= 128, CBRS_E_INVALID, "%s: n_users=%lld n_items=%d k=%d", who,
                 (long long)n_users, n_items, k);
    return CBRS_OK;
}

// Launches `excl` when the parameters carry exclusion lists, `plain` otherwise, with `smem` bytes of dynamic shared
// memory (at most smem_limit).  The attribute is set on every call: it belongs to the current device's context.
template <typename Params>
static int launch_catalog_scorer(void (*plain)(Params), void (*excl)(Params), const Params &p, unsigned grid,
                                 unsigned block, size_t smem, size_t smem_limit, cudaStream_t s, const char *who,
                                 const char *what) {
    CBRS_REQUIRE(smem <= smem_limit, CBRS_E_UNSUPPORTED, "%s: needs %zu bytes of shared memory", who, smem);
    auto kernel = p.excl_rowptr ? excl : plain;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));
    kernel<<<grid, block, smem, s>>>(p);
    CBRS_CHECK_LAUNCH(what);
    return CBRS_OK;
}

}  // namespace cbrs
