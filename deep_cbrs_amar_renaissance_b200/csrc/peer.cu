// Peer memory over NVLink / NVSwitch for the row-partitioned propagation (SURVEY 8e).
//
// The reference is single-process; this file belongs to the multi-GPU extension the north
// star asks for.  One process per GPU.  Every rank allocates the SAME set of buffers
// ("symmetric": same size, same layout), exports a CUDA IPC handle for each and maps its
// peers' copies.  The producing kernels (cbrs_dense_bcast / cbrs_spmm_csr_bcast) then store
// each finished output row into every rank's copy directly - the all-gather of a layer's
// operand happens inside the kernel that computes it, tile by tile, as plain st.global on
// peer-mapped addresses - and cbrs_peer_barrier closes the step: a one-CTA kernel that
// publishes an epoch number into every peer's flag array (st.release.sys after
// fence.acq_rel.sys) and spins (ld.acquire.sys) until every peer has published the same epoch
// into ours.  A stream-ordered barrier, no host involvement, no NCCL call on the data path.
#include "common.cuh"

#include <string.h>

namespace cbrs {

struct BarrierParams {
    unsigned long long *flags[CBRS_MAX_PEERS];  // flags[r] = rank r's array of CBRS_MAX_PEERS epochs
    int n_ranks;
    int me;
    unsigned long long epoch;
    unsigned long long timeout_ns;
    int *status;  // local: set to 1 if a peer did not arrive in time (the kernel then traps)
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__global__ void peer_barrier_kernel(const BarrierParams p) {
    const int t = threadIdx.x;
    if (t >= p.n_ranks) return;
    // everything this rank's earlier kernels stored (also into peer memory) is ordered before the flag
    __threadfence_system();
    st_release_sys(p.flags[t] + p.me, p.epoch);
    const unsigned long long t0 = globaltimer_ns();
    const unsigned long long *mine = p.flags[p.me] + t;
    while (ld_acquire_sys(mine) < p.epoch) {
        if (globaltimer_ns() - t0 > p.timeout_ns) {
            // a peer never arrived: the operand buffers the consumer kernels are about to gather from are only partly
            // written.  Record it and kill the stream (sticky launch failure) so that no later kernel can return
            // silently wrong embeddings; every following CUDA call of this process raises.
            *p.status = 1;
            __threadfence_system();
            __trap();
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_peer_alloc(size_t bytes, void **ptr_out) {
    CBRS_REQUIRE(ptr_out && bytes > 0, CBRS_E_INVALID, "peer_alloc: bad argument");
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        set_error("peer_alloc: cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
        return CBRS_E_CUDA;
    }
    e = cudaMemset(p, 0, bytes);
    if (e != cudaSuccess) {
        set_error("peer_alloc: cudaMemset: %s", cudaGetErrorString(e));
        cudaFree(p);
        return CBRS_E_CUDA;
    }
    *ptr_out = p;
    return CBRS_OK;
}

extern "C" int cbrs_peer_free(void *ptr) {
    if (!ptr) return CBRS_OK;
    cudaError_t e = cudaFree(ptr);
    if (e != cudaSuccess) {
        set_error("peer_free: %s", cudaGetErrorString(e));
        return CBRS_E_CUDA;
    }
    return CBRS_OK;
}

extern "C" int cbrs_peer_export(void *ptr, unsigned char *handle_host) {
    CBRS_REQUIRE(ptr && handle_host, CBRS_E_INVALID, "peer_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == CBRS_IPC_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
    if (e != cudaSuccess) {
        set_error("peer_export: cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
        return CBRS_E_CUDA;
    }
    memcpy(handle_host, &h, sizeof(h));
    return CBRS_OK;
}

extern "C" int cbrs_peer_open(const unsigned char *handle_host, void **ptr_out) {
    CBRS_REQUIRE(handle_host && ptr_out, CBRS_E_INVALID, "peer_open: null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle_host, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        set_error("peer_open: cudaIpcOpenMemHandle: %s", cudaGetErrorString(e));
        return CBRS_E_CUDA;
    }
    *ptr_out = p;
    return CBRS_OK;
}

extern "C" int cbrs_peer_close(void *ptr) {
    if (!ptr) return CBRS_OK;
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    if (e != cudaSuccess) {
        set_error("peer_close: %s", cudaGetErrorString(e));
        return CBRS_E_CUDA;
    }
    return CBRS_OK;
}

// Row block -> a mapped address (a peer's copy of a symmetric buffer, or its NVSwitch multicast mapping), coalesced:
// consecutive threads write consecutive 16-byte pieces of a row, so the fabric sees full 128-byte lines.
__global__ void push_rows_kernel(const float *__restrict__ src, int64_t lds, float *__restrict__ dst, int64_t ldd, int64_t m, int w4) {
    const int64_t total = m * w4;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / w4;
        const int c = (int)(e % w4) * 4;
        *reinterpret_cast<float4 *>(dst + r * ldd + c) = *reinterpret_cast<const float4 *>(src + r * lds + c);
    }
}
__global__ void push_rows_scalar_kernel(const float *__restrict__ src, int64_t lds, float *__restrict__ dst, int64_t ldd, int64_t m, int w) {
    const int64_t total = m * w;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x)
        dst[(e / w) * ldd + e % w] = src[(e / w) * lds + e % w];
}

extern "C" int cbrs_push_rows(const float *src, int64_t lds, void *dst, int64_t ldd, int64_t m, int32_t w, void *stream) {
    CBRS_REQUIRE(src && dst, CBRS_E_INVALID, "push_rows: null argument");
    CBRS_REQUIRE(m >= 0 && w > 0 && lds >= w && ldd >= w, CBRS_E_INVALID, "push_rows: bad shape");
    if (m == 0) return CBRS_OK;
    const bool vec = w % 4 == 0 && lds % 4 == 0 && ldd % 4 == 0 && ((uintptr_t)src & 15u) == 0 && ((uintptr_t)dst & 15u) == 0;
    const int64_t total = vec ? m * (w / 4) : m * (int64_t)w;
    const unsigned grid = (unsigned)(cdiv(total, 256) < 16 * kSMs ? cdiv(total, 256) : 16 * kSMs);
    if (vec)
        push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, lds, (float *)dst, ldd, m, w / 4);
    else
        push_rows_scalar_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, lds, (float *)dst, ldd, m, w);
    CBRS_CHECK_LAUNCH("push_rows");
    return CBRS_OK;
}

extern "C" int cbrs_peer_barrier(void *const *flags_peers_host, int n_ranks, int my_rank, uint64_t epoch,
                                 int32_t *status, double timeout_s, void *stream) {
    CBRS_REQUIRE(flags_peers_host && status, CBRS_E_INVALID, "peer_barrier: null argument");
    CBRS_REQUIRE(n_ranks >= 1 && n_ranks <= CBRS_MAX_PEERS && my_rank >= 0 && my_rank < n_ranks, CBRS_E_INVALID,
                 "peer_barrier: n_ranks=%d my_rank=%d", n_ranks, my_rank);
    BarrierParams p;
    for (int r = 0; r < CBRS_MAX_PEERS; ++r) p.flags[r] = r < n_ranks ? (unsigned long long *)flags_peers_host[r] : nullptr;
    for (int r = 0; r < n_ranks; ++r) CBRS_REQUIRE(p.flags[r], CBRS_E_INVALID, "peer_barrier: flags of rank %d are null", r);
    p.n_ranks = n_ranks;
    p.me = my_rank;
    p.epoch = epoch;
    p.timeout_ns = (unsigned long long)((timeout_s > 0 ? timeout_s : 30.0) * 1e9);
    p.status = status;
    peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(p);
    CBRS_CHECK_LAUNCH("peer_barrier");
    return CBRS_OK;
}
