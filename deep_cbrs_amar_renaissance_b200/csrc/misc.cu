// Small memory-bound helpers: layer reduction (row P5), row gather (S1/S3), the scaled
// synthetic graph generator (SURVEY 8d, config 5) and library plumbing.
#include "common.cuh"

#include <string.h>

namespace cbrs {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

constexpr int kMaxLayers = 16;
struct ReduceParams {
    const float *h[kMaxLayers];
    int64_t ld[kMaxLayers];
    float coef[kMaxLayers];
    int n_layers;
    float divide_by;
    int64_t n_rows;
    int32_t d;
    float *out;
    int64_t ldo;
};

// out = (sum_l coef_l * h_l) / divide_by, layers added in ascending l
// (/root/reference/src/layers/reduction.py:28-30,54-55: add_n then divide; sum(w^2 * h))
__global__ void reduce_layers_kernel(const ReduceParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_rows * p.d) return;
    const int64_t r = i / p.d;
    const int c = (int)(i % p.d);
    float acc = p.coef[0] * p.h[0][r * p.ld[0] + c];
    for (int l = 1; l < p.n_layers; ++l) acc += p.coef[l] * p.h[l][r * p.ld[l] + c];
    if (p.divide_by != 1.f) acc /= p.divide_by;
    p.out[r * p.ldo + c] = acc;
}

__global__ void gather_rows_kernel(const float *__restrict__ x, int64_t ldx, const int64_t *__restrict__ idx, int64_t m,
                                   int32_t d, float *__restrict__ out, int64_t ldo) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m * d) return;
    const int64_t r = i / d;
    const int c = (int)(i % d);
    out[r * ldo + c] = __ldg(x + idx[r] * ldx + c);
}

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// Integer-only generator (bit-identical on host and device).  Item popularity is a
// piecewise-uniform Zipf(1): octave j covers ranks [c*(2^j-1), c*(2^(j+1)-1)) and every
// octave carries the same mass, so the c hottest items each receive 1/(L*c) of the edges
// ("capped" head).  Ranks are scattered over item ids by a multiplicative bijection.
// Edges [edge_lo, edge_lo + m): entry k (edge edge_lo + k) goes to row[k], its reverse to row[m + k].
__global__ void synth_bipartite_kernel(int64_t n_users, int64_t n_items, int64_t edge_lo, int64_t m, uint64_t seed,
                                       uint64_t c, int levels, uint64_t mult, int32_t *__restrict__ row,
                                       int32_t *__restrict__ col) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int64_t e = edge_lo + k;
    const uint64_t h0 = splitmix64(seed ^ ((uint64_t)e * 0x2545F4914F6CDD1Dull));
    const uint64_t h1 = splitmix64(h0);
    const uint64_t h2 = splitmix64(h1);
    const int64_t u = (int64_t)(h0 % (uint64_t)n_users);
    const int lvl = (int)(h1 % (uint64_t)levels);
    const uint64_t span = c << lvl;
    const uint64_t rank = (span - c + (h2 % span)) % (uint64_t)n_items;
    const int64_t it = (int64_t)((rank * mult) % (uint64_t)n_items);
    row[k] = (int32_t)u;
    col[k] = (int32_t)(n_users + it);
    row[m + k] = (int32_t)(n_users + it);
    col[m + k] = (int32_t)u;
}

static uint64_t gcd64(uint64_t a, uint64_t b) { while (b) { uint64_t t = a % b; a = b; b = t; } return a; }

}  // namespace cbrs

using namespace cbrs;

extern "C" int cbrs_version(void) { return 100; }
extern "C" const char *cbrs_last_error(void) { return g_err; }

extern "C" int cbrs_check_device(void) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    CBRS_REQUIRE(e == cudaSuccess, CBRS_E_CUDA, "check_device: %s", cudaGetErrorString(e));
    int major = 0, minor = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    CBRS_REQUIRE(major == 10, CBRS_E_UNSUPPORTED, "check_device: compute capability %d.%d, kernels are built for sm_100a only",
                 major, minor);
    return CBRS_OK;
}

extern "C" int cbrs_reduce_layers(const float *const *h_host, const int64_t *ld_host, int32_t n_layers,
                                  const float *coef_host, float divide_by, int64_t n_rows, int32_t d, float *out,
                                  int64_t ldo, void *stream) {
    CBRS_REQUIRE(h_host && ld_host && out, CBRS_E_INVALID, "reduce_layers: null argument");
    CBRS_REQUIRE(n_layers >= 1 && n_layers <= kMaxLayers, CBRS_E_INVALID, "reduce_layers: n_layers=%d (max %d)", n_layers, kMaxLayers);
    CBRS_REQUIRE(n_rows >= 0 && d > 0 && ldo >= d && divide_by != 0.f, CBRS_E_INVALID, "reduce_layers: bad shape");
    if (n_rows == 0) return CBRS_OK;
    ReduceParams p;
    memset(&p, 0, sizeof(p));
    for (int l = 0; l < n_layers; ++l) {
        CBRS_REQUIRE(h_host[l] && ld_host[l] >= d, CBRS_E_INVALID, "reduce_layers: layer %d", l);
        p.h[l] = h_host[l];
        p.ld[l] = ld_host[l];
        p.coef[l] = coef_host ? coef_host[l] : 1.f;
    }
    p.n_layers = n_layers; p.divide_by = divide_by; p.n_rows = n_rows; p.d = d; p.out = out; p.ldo = ldo;
    reduce_layers_kernel<<<(unsigned)cdiv(n_rows * d, 256), 256, 0, (cudaStream_t)stream>>>(p);
    CBRS_CHECK_LAUNCH("reduce_layers");
    return CBRS_OK;
}

extern "C" int cbrs_gather_rows(const float *x, int64_t ldx, const int64_t *idx, int64_t m, int32_t d, float *out,
                                int64_t ldo, void *stream) {
    CBRS_REQUIRE(x && idx && out, CBRS_E_INVALID, "gather_rows: null argument");
    CBRS_REQUIRE(m >= 0 && d > 0 && ldx >= d && ldo >= d, CBRS_E_INVALID, "gather_rows: bad shape");
    if (m == 0) return CBRS_OK;
    gather_rows_kernel<<<(unsigned)cdiv(m * d, 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, idx, m, d, out, ldo);
    CBRS_CHECK_LAUNCH("gather_rows");
    return CBRS_OK;
}

extern "C" int cbrs_synth_bipartite(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed, int32_t *coo_row,
                                    int32_t *coo_col, void *stream) {
    return cbrs_synth_bipartite_ex(n_users, n_items, n_edges, seed, 1, coo_row, coo_col, stream);
}

extern "C" int cbrs_synth_bipartite_ex(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed, int scatter_items,
                                       int32_t *coo_row, int32_t *coo_col, void *stream) {
    CBRS_REQUIRE(coo_row && coo_col, CBRS_E_INVALID, "synth_bipartite: null argument");
    return cbrs_synth_bipartite_range(n_users, n_items, n_edges, seed, scatter_items, 0, n_edges, coo_row, coo_col, stream);
}

extern "C" int cbrs_synth_bipartite_range(int64_t n_users, int64_t n_items, int64_t n_edges, uint64_t seed,
                                          int scatter_items, int64_t edge_lo, int64_t edge_hi, int32_t *coo_row,
                                          int32_t *coo_col, void *stream) {
    CBRS_REQUIRE(n_users > 0 && n_items > 0 && n_edges >= 0 && n_users + n_items < ((int64_t)1 << 31), CBRS_E_INVALID,
                 "synth_bipartite: bad shape");
    CBRS_REQUIRE(0 <= edge_lo && edge_lo <= edge_hi && edge_hi <= n_edges, CBRS_E_INVALID,
                 "synth_bipartite: edge range [%lld, %lld) outside [0, %lld)", (long long)edge_lo, (long long)edge_hi,
                 (long long)n_edges);
    const int64_t m = edge_hi - edge_lo;
    if (m == 0) return CBRS_OK;
    CBRS_REQUIRE(coo_row && coo_col, CBRS_E_INVALID, "synth_bipartite: null argument");
    const uint64_t c = (uint64_t)(n_items / 1024 > 0 ? n_items / 1024 : 1);
    int levels = 1;
    while (c * ((1ull << levels) - 1) < (uint64_t)n_items) ++levels;
    uint64_t mult = 0x9E3779B1ull % (uint64_t)n_items;
    if (mult == 0) mult = 1;
    while (gcd64(mult, (uint64_t)n_items) != 1) ++mult;
    if (!scatter_items) mult = 1;  // item id = popularity rank: the hottest items are neighbours in id space
    synth_bipartite_kernel<<<(unsigned)cdiv(m, 256), 256, 0, (cudaStream_t)stream>>>(n_users, n_items, edge_lo, m, seed, c,
                                                                                   levels, mult, coo_row, coo_col);
    CBRS_CHECK_LAUNCH("synth_bipartite");
    return CBRS_OK;
}
