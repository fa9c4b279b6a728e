// lcp.cu -- K6: the LCP array and the permuted LCP array from the suffix array (DESIGN.md section 3, K6).
//
// Irreducible-PLCP method (Karkkainen, Manzini, Puglisi, "Permuted Longest-Common-Prefix Array", CPM 2009).  With
// Phi[SA[r]] = SA[r-1], position i is irreducible when i == 0, Phi[i] == 0, text[i-1] != text[Phi[i]-1], or i = SA[0];
// every other position has PLCP[i] = PLCP[i-1] - 1 (prepending a shared symbol to two adjacent suffixes keeps them
// adjacent).  That holds for any suffix order of the text, sentinel unique or not.  So only the irreducible values
// are computed by comparing text, and their sum is <= 2 n log2 n on every text; the rest follow from an inclusive
// max-scan of PLCP[i] + i, which is non-decreasing and constant across each run of reducible positions.
//
//   1. lcp_phi_kernel      one pass over SA: W[SA[r]] = SA[r-1] | IRR when irreducible (random 4-byte writes)
//   2. lcp_first_kernel    per irreducible i the first 32 symbols of (i, Phi[i]); a pair still equal goes to a list
//      lcp_round_kernel    round t compares the window [32 2^(t-1), 32 2^t) of every listed pair, one 8-byte word per
//                          item of a flat grid-stride loop (all pairs have the same window), the first mismatch by
//                          atomicMin into W[i]; lcp_compact_kernel keeps the pairs still equal.  The list count lives
//                          on the device and an empty round exits at once: the host launches a fixed number of
//                          rounds and does not wait.  Work <= 2 sum(irreducible lcp) + 32 #irreducible compares.
//   3. lcp_tile_max_kernel + seg_scan_kernel (the suffix-array build's tile scan) + lcp_apply_kernel: the max-scan
//   4. LCP[r] = PLCP[SA[r]] by hkcsa_gather_u32
//
// W is one uint32 per position: during step 1 Phi with the irreducible flag in bit 31 (values < 2^30); from step 2 on
// IRR | (PLCP[i] + i) at irreducible positions.  The pair lists are sized for a chunk of text positions: step 2 runs
// chunk by chunk, so a text with many long irreducible pairs never overflows them.
#include "common.cuh"
#include "prof.cuh"
#include "suffix_array.cuh"

namespace hkcsa {

constexpr uint32_t LCP_IRR = 0x80000000u;      // W word: irreducible position
constexpr uint32_t LCP_VAL = 0x7FFFFFFFu;
constexpr uint32_t LCP_NO_PRED = LCP_VAL;      // Phi of SA[0]: no predecessor, PLCP = 0 (positions are < 2^30)
constexpr uint32_t LCP_HEAD = 32;              // symbols compared by lcp_first_kernel
constexpr int LCP_THREADS = 256;
constexpr int LCP_IPT = 8;
constexpr int LCP_TILE = LCP_THREADS * LCP_IPT;
constexpr uint64_t LCP_CHUNK_MIN = 1ull << 22;  // positions per chunk of step 2: all of a text up to 4 M symbols,
constexpr uint64_t LCP_CHUNKS = 16;             // beyond that n / 16 (the lists then take n bytes)

// 8 bytes text[p .. p+8) as a little-endian word (p + 8 <= n): two aligned 8-byte loads and a funnel shift where
// both aligned words lie inside the text, single bytes at its two ends -- nothing outside [text, text + n) is read.
__device__ __forceinline__ uint64_t lcp_load8(const uint8_t *__restrict__ text, uint64_t n, uint64_t p)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(text + p);
    const uintptr_t base = a & ~(uintptr_t)7;
    const uint32_t sh = (uint32_t)(a & 7u) * 8u;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(text);
    if (base >= lo && base + 16 <= lo + n) {
        const uint64_t *w = reinterpret_cast<const uint64_t *>(base);
        const uint64_t w0 = __ldg(w);
        return sh ? (w0 >> sh) | (__ldg(w + 1) << (64u - sh)) : w0;
    }
    uint64_t v = 0;
    for (uint32_t b = 0; b < 8; ++b) v |= (uint64_t)text[p + b] << (8 * b);
    return v;
}

// index of the first k < len (len <= 8, a + len <= n, b + len <= n) with text[a+k] != text[b+k]; len when none
__device__ __forceinline__ uint32_t lcp_diff8(const uint8_t *__restrict__ text, uint64_t n, uint64_t a, uint64_t b,
                                              uint32_t len)
{
    if (len == 8) {
        const uint64_t x = lcp_load8(text, n, a) ^ lcp_load8(text, n, b);
        return x ? (uint32_t)(__ffsll((long long)x) - 1) >> 3 : 8u;
    }
    for (uint32_t k = 0; k < len; ++k)
        if (text[a + k] != text[b + k]) return k;
    return len;
}

// slot in a list whose count is *count, one atomic per group of lanes that append together
__device__ __forceinline__ uint32_t lcp_append_slot(uint32_t *count)
{
    const uint32_t m = __activemask();
    const uint32_t leader = __ffs(m) - 1;
    uint32_t base = 0;
    if (lane_id() == leader) base = atomicAdd(count, (uint32_t)__popc(m));
    base = __shfl_sync(m, base, leader);
    return base + __popc(m & lanemask_lt());
}

__global__ void __launch_bounds__(LCP_THREADS)
lcp_phi_kernel(const uint8_t *__restrict__ text, const uint32_t *__restrict__ sa, uint32_t n, uint32_t *__restrict__ W)
{
    const uint32_t r = blockIdx.x * LCP_THREADS + threadIdx.x;
    if (r >= n) return;
    const uint32_t i = sa[r];
    if (r == 0) { W[i] = LCP_IRR | LCP_NO_PRED; return; }
    const uint32_t j = sa[r - 1];
    const bool irr = i == 0 || j == 0 || text[i - 1] != text[j - 1];
    W[i] = irr ? (LCP_IRR | j) : j;
}

// irreducible positions of [c0, c1): the first LCP_HEAD symbols.  Finished: W[i] = IRR | (i + lcp).  Still equal:
// W[i] = IRR | (i + cap), cap = symbols left in the shorter suffix, and (i, Phi[i]) goes to the list.
__global__ void __launch_bounds__(LCP_THREADS)
lcp_first_kernel(const uint8_t *__restrict__ text, uint32_t n, uint32_t *__restrict__ W, uint32_t c0, uint32_t c1,
                 uint2 *__restrict__ list, uint32_t *__restrict__ count)
{
    for (uint32_t i = c0 + blockIdx.x * LCP_THREADS + threadIdx.x; i < c1; i += gridDim.x * LCP_THREADS) {
        const uint32_t w = W[i];
        if (!(w & LCP_IRR)) continue;
        const uint32_t j = w & LCP_VAL;
        uint32_t v = i;
        if (j != LCP_NO_PRED) {
            const uint32_t cap = n - max(i, j);
            const uint32_t lim = min(cap, LCP_HEAD);
            uint32_t l = 0;
            while (l < lim) {
                const uint32_t len = min(8u, lim - l);
                const uint32_t k = lcp_diff8(text, n, (uint64_t)i + l, (uint64_t)j + l, len);
                l += k;
                if (k < len) break;
            }
            v = i + l;
            if (l == LCP_HEAD && cap > LCP_HEAD) {
                v = i + cap;
                list[lcp_append_slot(count)] = make_uint2(i, j);
            }
        }
        W[i] = LCP_IRR | v;
    }
}

// one round: the window [start, start + 8 << log_words) of every listed pair; zeroes the count the following
// compaction fills (*next_count) before it looks at its own
__global__ void __launch_bounds__(LCP_THREADS)
lcp_round_kernel(const uint8_t *__restrict__ text, uint32_t n, const uint2 *__restrict__ list,
                 const uint32_t *__restrict__ count, uint32_t *__restrict__ next_count, uint32_t *__restrict__ W,
                 uint32_t start, uint32_t log_words)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) *next_count = 0;
    const uint32_t m = *count;
    if (m == 0) return;
    const uint64_t items = (uint64_t)m << log_words, mask = (1ull << log_words) - 1;
    for (uint64_t t = (uint64_t)blockIdx.x * LCP_THREADS + threadIdx.x; t < items; t += (uint64_t)gridDim.x * LCP_THREADS) {
        const uint2 e = list[t >> log_words];
        const uint32_t cap = n - max(e.x, e.y);
        const uint64_t o = start + ((t & mask) << 3);
        if (o >= cap) continue;
        const uint32_t len = (uint32_t)min((uint64_t)8, cap - o);
        const uint32_t k = lcp_diff8(text, n, e.x + o, e.y + o, len);
        if (k < len) atomicMin(&W[e.x], LCP_IRR | (uint32_t)(e.x + o + k));
    }
}

// pairs with no mismatch so far whose shorter suffix goes on past `end` stay for the next round
__global__ void __launch_bounds__(LCP_THREADS)
lcp_compact_kernel(uint32_t n, const uint2 *__restrict__ list, const uint32_t *__restrict__ count,
                   const uint32_t *__restrict__ W, uint64_t end, uint2 *__restrict__ next, uint32_t *__restrict__ next_count)
{
    const uint32_t m = *count;
    for (uint32_t p = blockIdx.x * LCP_THREADS + threadIdx.x; p < m; p += gridDim.x * LCP_THREADS) {
        const uint2 e = list[p];
        const uint32_t cap = n - max(e.x, e.y);
        if (cap > end && W[e.x] == (LCP_IRR | (e.x + cap))) next[lcp_append_slot(next_count)] = e;
    }
}

// the max-scan input: PLCP[i] + i at irreducible positions, 0 elsewhere
__device__ __forceinline__ uint32_t lcp_scan_value(uint32_t w) { return (w & LCP_IRR) ? (w & LCP_VAL) : 0u; }

__device__ __forceinline__ void lcp_load_tile(const uint32_t *__restrict__ W, uint32_t n, uint32_t i0,
                                              uint32_t (&w)[LCP_IPT])
{
    if (i0 + LCP_IPT <= n) {
        const uint4 *v = reinterpret_cast<const uint4 *>(W + i0);      // i0 is a multiple of 8, W 256-byte aligned
        const uint4 a = v[0], b = v[1];
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
#pragma unroll
        for (int e = 0; e < LCP_IPT; ++e) w[e] = (i0 + e < n) ? W[i0 + e] : 0u;
    }
}

__global__ void __launch_bounds__(LCP_THREADS)
lcp_tile_max_kernel(const uint32_t *__restrict__ W, uint32_t n, uint32_t *__restrict__ agg)
{
    __shared__ uint32_t s_w[LCP_THREADS / 32];
    uint32_t w[LCP_IPT];
    lcp_load_tile(W, n, blockIdx.x * LCP_TILE + threadIdx.x * LCP_IPT, w);
    uint32_t m = 0;
#pragma unroll
    for (int e = 0; e < LCP_IPT; ++e) m = max(m, lcp_scan_value(w[e]));
    m = __reduce_max_sync(0xffffffffu, m);
    if (lane_id() == 0) s_w[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < LCP_THREADS / 32; ++k) m = max(m, s_w[k]);
        agg[blockIdx.x] = m;
    }
}

// out[i] = (inclusive max-scan of the values)[i] - i; agg = the exclusive scan of the tile maxima.  stats (may be
// null): += (irreducible positions, sum of their values)
__global__ void __launch_bounds__(LCP_THREADS)
lcp_apply_kernel(const uint32_t *__restrict__ W, uint32_t n, const uint32_t *__restrict__ agg, uint32_t *out,
                 unsigned long long *__restrict__ stats)
{
    __shared__ uint32_t s_w[LCP_THREADS / 32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t i0 = blockIdx.x * LCP_TILE + threadIdx.x * LCP_IPT;
    uint32_t w[LCP_IPT];
    lcp_load_tile(W, n, i0, w);
    uint32_t th = 0;
#pragma unroll
    for (int e = 0; e < LCP_IPT; ++e) th = max(th, lcp_scan_value(w[e]));
    const uint32_t incl = warp_incl_max(th);
    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t run = agg[blockIdx.x];
    for (uint32_t k = 0; k < warp; ++k) run = max(run, s_w[k]);
    if (lane) run = max(run, up);
    uint32_t cnt = 0;
    unsigned long long sum = 0;
#pragma unroll
    for (int e = 0; e < LCP_IPT; ++e) {
        const uint32_t i = i0 + e;
        const uint32_t v = lcp_scan_value(w[e]);
        run = max(run, v);
        if (i < n) {
            out[i] = run - i;
            if (w[e] & LCP_IRR) { ++cnt; sum += v - i; }
        }
    }
    if (stats) {
        cnt = __reduce_add_sync(0xffffffffu, cnt);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, o);
        if (lane == 0 && cnt) {
            atomicAdd(&stats[0], (unsigned long long)cnt);
            atomicAdd(&stats[1], sum);
        }
    }
}

__global__ void plcp_bits_kernel(const uint32_t *__restrict__ plcp, uint32_t n, uint8_t *__restrict__ bits)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i >= n) return;
    const uint64_t p = (uint64_t)plcp[i] + 2ull * i;
    if (p < 2ull * n) bits[p] = 1;            // a PLCP value is < n - i; anything else is not a PLCP array
}

static uint64_t lcp_chunk(uint64_t n)
{
    return n <= LCP_CHUNK_MIN ? n : std::max(LCP_CHUNK_MIN, (n + LCP_CHUNKS - 1) / LCP_CHUNKS);
}

struct LcpBuffers {
    uint32_t *W, *agg, *keep, *counts;   // counts: [0, 1] list counts, [2] scan total (unused)
    unsigned long long *stats;
    uint2 *list[2];
};
static LcpBuffers carve_lcp(Carver &c, uint64_t n)
{
    LcpBuffers b;
    const uint64_t tiles = (n + LCP_TILE - 1) / LCP_TILE, chunk = lcp_chunk(n);
    b.W = c.take<uint32_t>(n);
    b.agg = c.take<uint32_t>(tiles);
    b.keep = c.take<uint32_t>(tiles);
    b.counts = c.take<uint32_t>(4);
    b.stats = c.take<unsigned long long>(2);
    b.list[0] = c.take<uint2>(chunk);
    b.list[1] = c.take<uint2>(chunk);
    return b;
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" size_t hkcsa_lcp_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    carve_lcp(c, n ? n : 1);
    return c.total();
}

extern "C" int hkcsa_lcp_build(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t *d_lcp,
                               uint32_t *d_plcp, void *d_scratch, size_t scratch_bytes, uint64_t *h_stats, void *stream)
{
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    if (h_stats) h_stats[0] = h_stats[1] = 0;
    if (n == 0) return HKCSA_OK;
    HK_REQUIRE(d_text && d_sa && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(d_lcp || d_plcp, HKCSA_EINVAL, "no output: d_lcp and d_plcp are both NULL");
    Carver c(d_scratch);
    LcpBuffers B = carve_lcp(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "lcp scratch too small");
    cudaStream_t st = as_stream(stream);
    const uint32_t n32 = (uint32_t)n;
    const uint32_t tiles = (uint32_t)((n + LCP_TILE - 1) / LCP_TILE);
    const uint64_t chunk = lcp_chunk(n);
    const uint32_t grid = (uint32_t)num_sms() * 8u;
    uint32_t rounds = 0;                                       // the window of the last round reaches past n
    while (((uint64_t)LCP_HEAD << rounds) < n) ++rounds;
    prof::Scope ps(st, prof::OTHER, n * 26ull);
    if (h_stats) HK_CUDA(cudaMemsetAsync(B.stats, 0, 2 * sizeof(unsigned long long), st));
    HK_CUDA(cudaMemsetAsync(B.keep, 0, (size_t)tiles * sizeof(uint32_t), st));

    lcp_phi_kernel<<<(n32 + LCP_THREADS - 1) / LCP_THREADS, LCP_THREADS, 0, st>>>(d_text, d_sa, n32, B.W);
    HK_LAUNCH_CHECK();
    for (uint64_t c0 = 0; c0 < n; c0 += chunk) {
        const uint32_t c1 = (uint32_t)std::min(n, c0 + chunk);
        HK_CUDA(cudaMemsetAsync(B.counts, 0, 2 * sizeof(uint32_t), st));
        lcp_first_kernel<<<(uint32_t)std::min<uint64_t>(grid, (c1 - c0 + LCP_THREADS - 1) / LCP_THREADS), LCP_THREADS,
                           0, st>>>(d_text, n32, B.W, (uint32_t)c0, c1, B.list[0], B.counts);
        HK_LAUNCH_CHECK();
        for (uint32_t t = 1, cur = 0; t <= rounds; ++t, cur ^= 1) {
            const uint64_t start = (uint64_t)LCP_HEAD << (t - 1), end = (uint64_t)LCP_HEAD << t;
            lcp_round_kernel<<<grid, LCP_THREADS, 0, st>>>(d_text, n32, B.list[cur], B.counts + cur,
                                                            B.counts + (cur ^ 1), B.W, (uint32_t)start, t + 1);
            HK_LAUNCH_CHECK();
            if (t == rounds) break;                            // nothing outlives the last window
            lcp_compact_kernel<<<grid, LCP_THREADS, 0, st>>>(n32, B.list[cur], B.counts + cur, B.W, end,
                                                              B.list[cur ^ 1], B.counts + (cur ^ 1));
            HK_LAUNCH_CHECK();
        }
    }
    uint32_t *plcp = d_plcp ? d_plcp : B.W;                    // PLCP only for the gather: in place over W
    lcp_tile_max_kernel<<<tiles, LCP_THREADS, 0, st>>>(B.W, n32, B.agg);
    HK_LAUNCH_CHECK();
    seg_scan_kernel<<<1, 1024, 0, st>>>(B.agg, B.keep, tiles, B.counts + 2);
    HK_LAUNCH_CHECK();
    lcp_apply_kernel<<<tiles, LCP_THREADS, 0, st>>>(B.W, n32, B.agg, plcp, h_stats ? B.stats : nullptr);
    HK_LAUNCH_CHECK();
    if (d_lcp) {
        const int rc = hkcsa_gather_u32(plcp, d_sa, n, d_lcp, stream);
        if (rc != HKCSA_OK) return rc;
    }
    if (h_stats) {
        unsigned long long s[2];
        HK_CUDA(cudaMemcpyAsync(s, B.stats, sizeof(s), cudaMemcpyDeviceToHost, st));
        HK_CUDA(cudaStreamSynchronize(st));
        h_stats[0] = s[0];
        h_stats[1] = s[1];
    }
    return HKCSA_OK;
}

extern "C" int hkcsa_plcp_bits(const uint32_t *d_plcp, uint64_t n, uint8_t *d_bits, void *stream)
{
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    if (n == 0) return HKCSA_OK;
    HK_REQUIRE(d_plcp && d_bits, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemsetAsync(d_bits, 0, 2 * n, st));
    plcp_bits_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, st>>>(d_plcp, (uint32_t)n, d_bits);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
