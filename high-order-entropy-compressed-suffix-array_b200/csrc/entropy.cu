// entropy.cu -- k-th order empirical entropy H_k from the suffix array (SURVEY.md section 8f, row 2).
//
// Replaces calculate_high_order_entropy (reference csa/high_order_entropy.py:4-32) for k >= 1:
//     H_k = (1/n) * sum over k-gram contexts w of |w|_next * H_0(symbols following w)
//         = (1/n) * ( sum_w T_w log2 T_w  -  sum_{wc} c_{wc} log2 c_{wc} )
// where T_w counts the windows text[i : i+k+1], i in [0, n-k), whose first k symbols are w, and c_{wc} those that
// read wc -- the reference normalises by n, not n-k (:30).  The windows sharing a (k+1)-gram are exactly a run of
// adjacent suffixes in the suffix array, so with the suffix array at hand (the index build has it) no k-gram
// keys are packed or sorted and k is not limited by a key width: one pass flags the run heads by comparing each
// suffix's first k (+1) symbols with its predecessor's, a scan numbers them, and the run lengths feed two fp64
// sums that are reduced in a fixed order (bit-reproducible).
#include "common.cuh"
#include "prof.cuh"
#include <math.h>

namespace hkcsa {

constexpr int HK_THREADS = 256;
constexpr int HK_IPT = 8;
constexpr int HK_TILE = HK_THREADS * HK_IPT;

// do the suffixes a and b (both with at least `len` symbols) agree on their first `len` symbols?
__device__ __forceinline__ bool same_prefix(const uint8_t *__restrict__ text, uint64_t a, uint64_t b, uint32_t len)
{
    for (uint32_t q = 0; q < len; ++q)
        if (text[a + q] != text[b + q]) return false;
    return true;
}

// flags of entry j: bit 0 = valid (the suffix has k+1 symbols: it is a window), bit 1 = head of a (k+1)-gram run,
// bit 2 = head of a k-gram run (among valid entries)
__device__ __forceinline__ uint32_t hk_flags(const uint8_t *__restrict__ text, uint64_t n, const uint32_t *__restrict__ sa,
                                             uint64_t j, uint32_t k)
{
    const uint64_t a = sa[j];
    if (a + k >= n) return 0u;
    if (j == 0) return 7u;
    const uint64_t b = sa[j - 1];
    const bool prev_valid = b + k < n;
    // a suffix shorter than k+1 symbols cannot share k+1 symbols; one of exactly k symbols (the context alone, it
    // sorts first in its context's range) does not count as a window
    if (!prev_valid) return 7u;
    if (!same_prefix(text, a, b, k)) return 7u;
    return text[a + k] != text[b + k] ? 3u : 1u;
}

__device__ __forceinline__ uint32_t block_excl_sum3(uint32_t v0, uint32_t v1, uint32_t v2, uint32_t (&tot)[3],
                                                    uint32_t &e1, uint32_t &e2)
{
    __shared__ uint32_t s_w[3][HK_THREADS / 32];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t t0, t1, t2;
    const uint32_t x0 = warp_excl_sum(v0, t0), x1 = warp_excl_sum(v1, t1), x2 = warp_excl_sum(v2, t2);
    if (lane == 31) { s_w[0][warp] = t0; s_w[1][warp] = t1; s_w[2][warp] = t2; }
    __syncthreads();
    uint32_t p0 = 0, p1 = 0, p2 = 0;
    tot[0] = tot[1] = tot[2] = 0;
    for (uint32_t w = 0; w < HK_THREADS / 32; ++w) {
        if (w < warp) { p0 += s_w[0][w]; p1 += s_w[1][w]; p2 += s_w[2][w]; }
        tot[0] += s_w[0][w]; tot[1] += s_w[1][w]; tot[2] += s_w[2][w];
    }
    __syncthreads();
    e1 = x1 + p1;
    e2 = x2 + p2;
    return x0 + p0;
}

// pass 1: per-tile counts of (valid, (k+1)-gram heads, k-gram heads); the flags are kept (one byte per entry)
__global__ void __launch_bounds__(HK_THREADS)
hk_count_kernel(const uint8_t *__restrict__ text, uint64_t n, const uint32_t *__restrict__ sa, uint32_t k,
                uint8_t *__restrict__ flags, uint32_t *__restrict__ tile_cnt /* [3][tiles] */, uint32_t tiles)
{
    const uint64_t j0 = (uint64_t)blockIdx.x * HK_TILE + (uint64_t)threadIdx.x * HK_IPT;
    uint32_t c0 = 0, c1 = 0, c2 = 0;
    uint64_t packed = 0;
#pragma unroll
    for (int e = 0; e < HK_IPT; ++e) {
        const uint64_t j = j0 + e;
        const uint32_t f = j < n ? hk_flags(text, n, sa, j, k) : 0u;
        packed |= (uint64_t)f << (8 * e);
        c0 += f & 1u; c1 += (f >> 1) & 1u; c2 += (f >> 2) & 1u;
    }
    if (j0 + HK_IPT <= n) *reinterpret_cast<uint64_t *>(flags + j0) = packed;        // flags is 8-byte aligned
    else for (int e = 0; e < HK_IPT && j0 + e < n; ++e) flags[j0 + e] = (uint8_t)(packed >> (8 * e));
    uint32_t tot[3], e1, e2;
    block_excl_sum3(c0, c1, c2, tot, e1, e2);
    if (threadIdx.x == 0) {
        tile_cnt[blockIdx.x] = tot[0];
        tile_cnt[tiles + blockIdx.x] = tot[1];
        tile_cnt[2 * tiles + blockIdx.x] = tot[2];
    }
}

// single CTA: exclusive scan (64-bit running totals kept as uint32 -- n <= HKCSA_MAX_N) of each of the 3 rows
__global__ void __launch_bounds__(1024)
hk_scan_kernel(uint32_t *__restrict__ tile_cnt, uint32_t tiles, uint32_t *__restrict__ totals /* [3] */)
{
    for (int row = 0; row < 3; ++row) {
        uint32_t *c = tile_cnt + (size_t)row * tiles;
        const uint32_t t = block_excl_scan_carried(tiles, 0u, Plus(), [&](uint32_t i) { return c[i]; },
                                                   [&](uint32_t i, uint32_t p) { c[i] = p; });
        if (threadIdx.x == 0) totals[row] = t;
    }
}

// pass 2: every run head stores the number of valid entries before it: H1[r] for the r-th (k+1)-gram run, H0[r]
// for the r-th k-gram run
__global__ void __launch_bounds__(HK_THREADS)
hk_heads_kernel(const uint8_t *__restrict__ flags, uint64_t n, const uint32_t *__restrict__ tile_base, uint32_t tiles,
                uint32_t *__restrict__ H1, uint32_t *__restrict__ H0)
{
    const uint64_t j0 = (uint64_t)blockIdx.x * HK_TILE + (uint64_t)threadIdx.x * HK_IPT;
    uint32_t f[HK_IPT];
    uint32_t c0 = 0, c1 = 0, c2 = 0;
#pragma unroll
    for (int e = 0; e < HK_IPT; ++e) {
        f[e] = (j0 + e < n) ? flags[j0 + e] : 0u;
        c0 += f[e] & 1u; c1 += (f[e] >> 1) & 1u; c2 += (f[e] >> 2) & 1u;
    }
    uint32_t tot[3], e1, e2;
    uint32_t v = block_excl_sum3(c0, c1, c2, tot, e1, e2) + tile_base[blockIdx.x];
    uint32_t r1 = e1 + tile_base[tiles + blockIdx.x], r0 = e2 + tile_base[2 * tiles + blockIdx.x];
#pragma unroll
    for (int e = 0; e < HK_IPT; ++e) {
        if (f[e] & 2u) H1[r1++] = v;
        if (f[e] & 4u) H0[r0++] = v;
        v += f[e] & 1u;
    }
}

// pass 3: partial[block] = sum over this block's runs of c * log2(c), c = H[r+1] - H[r] (the last run ends at
// `n_valid`); summed inside the block in a fixed tree order
__global__ void __launch_bounds__(HK_THREADS)
hk_sum_kernel(const uint32_t *__restrict__ H, uint32_t runs, uint32_t n_valid, double *__restrict__ partial)
{
    __shared__ double s_p[HK_THREADS];
    double acc = 0.0;
    const uint64_t r0 = (uint64_t)blockIdx.x * HK_TILE;
    for (int e = 0; e < HK_IPT; ++e) {
        const uint64_t r = r0 + (uint64_t)e * HK_THREADS + threadIdx.x;
        if (r < runs) {
            const uint32_t c = (r + 1 < runs ? H[r + 1] : n_valid) - H[r];
            if (c > 1) acc += (double)c * log2((double)c);
        }
    }
    s_p[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t s = HK_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) s_p[threadIdx.x] += s_p[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = s_p[0];
}

// single CTA: out = sum of partial[0 .. count) in index order per thread, then a fixed tree
__global__ void __launch_bounds__(HK_THREADS)
hk_final_kernel(const double *__restrict__ partial, uint32_t count, double *__restrict__ out)
{
    __shared__ double s_p[HK_THREADS];
    double acc = 0.0;
    for (uint32_t i = threadIdx.x; i < count; i += HK_THREADS) acc += partial[i];
    s_p[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t s = HK_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) s_p[threadIdx.x] += s_p[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = s_p[0];
}

struct HkBuffers {
    uint8_t *flags;
    uint32_t *tile_cnt, *totals, *H1, *H0;
    double *partial, *out;
};
static HkBuffers carve_hk(Carver &c, uint64_t n)
{
    HkBuffers b;
    const uint64_t tiles = (n + HK_TILE - 1) / HK_TILE + 1;
    b.flags = c.take<uint8_t>(n + 8);
    b.tile_cnt = c.take<uint32_t>(3 * tiles);
    b.totals = c.take<uint32_t>(4);
    b.H1 = c.take<uint32_t>(n + 1);
    b.H0 = c.take<uint32_t>(n + 1);
    b.partial = c.take<double>(tiles);
    b.out = c.take<double>(2);
    return b;
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" size_t hkcsa_entropy_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    carve_hk(c, n ? n : 1);
    return c.total();
}

// h_out[0] = sum over k-gram contexts of T log2 T, h_out[1] = sum over (k+1)-grams of c log2 c, h_out[2] = number
// of windows (n - k), h_out[3] = distinct contexts, h_out[4] = distinct (k+1)-grams.  H_k = (h_out[0] - h_out[1]) / n.
extern "C" int hkcsa_entropy_from_sa(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t k, double *h_out,
                                     void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(h_out != nullptr, HKCSA_EINVAL, "null pointer");
    for (int i = 0; i < 5; ++i) h_out[i] = 0.0;
    HK_REQUIRE(k >= 1, HKCSA_EINVAL, "k must be >= 1 (H_0 follows from the byte histogram)");
    if (n <= k) return HKCSA_OK;                   // calculate_high_order_entropy returns 0 (:17-18)
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    HK_REQUIRE(d_text && d_sa && d_scratch, HKCSA_EINVAL, "null pointer");
    Carver c(d_scratch);
    HkBuffers B = carve_hk(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "entropy scratch too small");
    cudaStream_t st = as_stream(stream);
    const uint32_t tiles = (uint32_t)((n + HK_TILE - 1) / HK_TILE);
    prof::Scope ps(st, prof::OTHER, n * (4 + 2ull * (k + 1) + 2));
    hk_count_kernel<<<tiles, HK_THREADS, 0, st>>>(d_text, n, d_sa, k, B.flags, B.tile_cnt, tiles);
    HK_LAUNCH_CHECK();
    hk_scan_kernel<<<1, 1024, 0, st>>>(B.tile_cnt, tiles, B.totals);
    HK_LAUNCH_CHECK();
    hk_heads_kernel<<<tiles, HK_THREADS, 0, st>>>(B.flags, n, B.tile_cnt, tiles, B.H1, B.H0);
    HK_LAUNCH_CHECK();
    uint32_t h_tot[3];
    HK_CUDA(cudaMemcpyAsync(h_tot, B.totals, sizeof(h_tot), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    const uint32_t n_valid = h_tot[0], runs1 = h_tot[1], runs0 = h_tot[2];
    double h_sums[2] = {0.0, 0.0};
    const uint32_t *Hs[2] = {B.H0, B.H1};
    const uint32_t runs[2] = {runs0, runs1};
    for (int which = 0; which < 2; ++which) {
        if (runs[which] == 0) continue;
        const uint32_t blocks = (runs[which] + HK_TILE - 1) / HK_TILE;
        hk_sum_kernel<<<blocks, HK_THREADS, 0, st>>>(Hs[which], runs[which], n_valid, B.partial);
        HK_LAUNCH_CHECK();
        hk_final_kernel<<<1, HK_THREADS, 0, st>>>(B.partial, blocks, B.out + which);
        HK_LAUNCH_CHECK();
    }
    HK_CUDA(cudaMemcpyAsync(h_sums, B.out, sizeof(h_sums), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    h_out[0] = runs0 ? h_sums[0] : 0.0;
    h_out[1] = runs1 ? h_sums[1] : 0.0;
    h_out[2] = (double)n_valid;
    h_out[3] = (double)runs0;
    h_out[4] = (double)runs1;
    return HKCSA_OK;
}
