// suffix_array.cu -- K1: suffix-array construction by prefix doubling.
//
// Replaces build_suffix_array (reference csa/suffix_array.py:131-134): the
// permutation that sorts all suffixes in byte order with a proper prefix first.
//
// Round 0 packs the first k0 symbols of every suffix (dense codes of b bits,
// 0 = "past the end", so shorter suffixes sort first) into one 64-bit key and
// radix-sorts (key, position).  Equal keys form groups; a suffix's rank is the
// SA position where its group starts.  Round r (depth h = k0 * 2^(r-1)) takes
// only the suffixes whose group is not yet a singleton, keys them with
// (group start, rank[i + h] + 1) -- 0 when i + h >= n -- sorts, and refines.
// Suffixes that became unique leave the working set (their SA slot is final).
#include "common.cuh"
#include "prof.cuh"
#include "radix_sort.cuh"
#include "suffix_array.cuh"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

namespace hkcsa {

static void alpha_assign(const double *cum, const int *item, int lo, int hi, uint32_t code, int len, AlphaCode &ac,
                         int &max_len)
{
    if (hi - lo == 1) {
        ac.code[item[lo]] = code;
        ac.len[item[lo]] = (uint8_t)std::max(len, 1);
        max_len = std::max(max_len, std::max(len, 1));
        return;
    }
    // split where the two halves weigh most alike
    int best = lo + 1;
    double best_d = 1e300;
    for (int sp = lo + 1; sp < hi; ++sp) {
        const double d = fabs((cum[sp] - cum[lo]) - (cum[hi] - cum[sp]));
        if (d < best_d) { best_d = d; best = sp; }
    }
    alpha_assign(cum, item, lo, best, code << 1, len + 1, ac, max_len);
    alpha_assign(cum, item, best, hi, (code << 1) | 1u, len + 1, ac, max_len);
}

// returns false when the code would be degenerate (then the caller keeps fixed-width codes)
bool build_alpha_code(const uint64_t *h_hist, AlphaCode &ac, double &avg_len, int &max_len)
{
    int item[257];
    double w[257], cum[258];
    int m = 0;
    double total = 0;
    for (int ch = 0; ch < 256; ++ch) total += (double)h_hist[ch];
    item[m] = 256; w[m] = 0; ++m;                       // past-the-end sorts first
    for (int ch = 0; ch < 256; ++ch)
        if (h_hist[ch]) { item[m] = ch; w[m] = (double)h_hist[ch]; ++m; }
    const double smooth = total / (8.0 * m) + 1.0;      // bounds the depth of rare symbols
    cum[0] = 0;
    for (int i = 0; i < m; ++i) cum[i + 1] = cum[i] + w[i] + smooth;
    for (int i = 0; i < 257; ++i) { ac.code[i] = 0; ac.len[i] = 1; }
    max_len = 0;
    if (m == 1) { ac.code[256] = 0; ac.len[256] = 1; max_len = 1; avg_len = 1; return true; }
    alpha_assign(cum, item, 0, m, 0u, 0, ac, max_len);
    if (max_len > 24) return false;
    avg_len = 0;
    for (int i = 1; i < m; ++i) avg_len += w[i] * ac.len[item[i]];
    avg_len = total > 0 ? avg_len / total : 1.0;
    return true;
}

// ---------------------------------------------------------------- byte histogram
__global__ void byte_hist_kernel(const uint8_t *__restrict__ text, uint64_t n, unsigned long long *__restrict__ ghist)
{
    __shared__ uint32_t s_h[8][256];   // one private histogram per warp
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < 8 * 256; i += blockDim.x) (&s_h[0][0])[i] = 0;
    __syncthreads();
    // 16-byte vector loads over the aligned middle; CTA 0 takes the ragged ends
    const uint64_t mis = (16 - (reinterpret_cast<uintptr_t>(text) & 15)) & 15;
    const uint64_t pre = mis < n ? mis : n;
    const uint64_t nvec = (n - pre) / 16;
    const uint4 *v = reinterpret_cast<const uint4 *>(text + pre);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + tid; i < nvec; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint4 q = v[i];
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_h[warp][w[j] & 0xFFu], 1u);
            atomicAdd(&s_h[warp][(w[j] >> 8) & 0xFFu], 1u);
            atomicAdd(&s_h[warp][(w[j] >> 16) & 0xFFu], 1u);
            atomicAdd(&s_h[warp][w[j] >> 24], 1u);
        }
    }
    if (blockIdx.x == 0) {
        for (uint64_t i = tid; i < pre; i += blockDim.x) atomicAdd(&s_h[warp][text[i]], 1u);
        for (uint64_t i = pre + nvec * 16 + tid; i < n; i += blockDim.x) atomicAdd(&s_h[warp][text[i]], 1u);
    }
    __syncthreads();
    if (tid < 256) {
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_h[w][tid];
        if (s) atomicAdd(&ghist[tid], (unsigned long long)s);
    }
}

cudaError_t byte_hist(const uint8_t *d_text, uint64_t n, uint64_t *d_hist, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(d_hist, 0, 256 * sizeof(uint64_t), st);
    if (e != cudaSuccess || n == 0) return e;
    const int blocks = (int)std::min<uint64_t>((n + 65535) / 65536, (uint64_t)num_sms() * 4);
    prof::Scope ps(st, prof::BYTE_HIST, n);
    byte_hist_kernel<<<std::max(blocks, 1), 256, 0, st>>>(d_text, n, reinterpret_cast<unsigned long long *>(d_hist));
    return cudaGetLastError();
}

// sampled k-gram histogram: CTA b counts the grams of tile b * stride (2048 positions) with global atomics
__global__ void __launch_bounds__(PACK_THREADS)
gram_hist_kernel(const uint8_t *__restrict__ text, uint32_t n, GramCode gc, uint32_t stride, uint32_t *__restrict__ gh)
{
    __shared__ uint8_t s_digit[256];
    __shared__ __align__(8) uint8_t s_dig[PACK_TILE + 16];
    const uint32_t tid = threadIdx.x;
    s_digit[tid] = gc.digit[tid];
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * stride * PACK_TILE;
    const bool aligned8 = (reinterpret_cast<uintptr_t>(text) & 7) == 0;
    const uint64_t p0 = base + (uint64_t)tid * PACK_IPT;
    reinterpret_cast<uint2 *>(s_dig)[tid] = GramKeys::digits8(s_digit, text, n, p0, aligned8);
    if (tid < 2) reinterpret_cast<uint2 *>(s_dig)[PACK_THREADS + tid] = GramKeys::digits8(s_digit, text, n, base + PACK_TILE + tid * 8u, aligned8);
    __syncthreads();
    uint32_t g[8];
    GramKeys::roll8(s_dig, tid * PACK_IPT, gc.k, gc.B, gc.pw, g);
#pragma unroll
    for (int e = 0; e < 8; ++e)
        if (p0 + e < n) atomicAdd(&gh[g[e]], 1u);
}

// Weights w[g] = 16 * count + smooth (smooth = max(1, samples / G): the unseen grams together weigh 1/16 of the seen
// ones, which bounds every code length by log2(17 G) + 2 <= 23 bits).  CTA c scans chunk c of 4096 grams: cum[] =
// exclusive prefix sums inside the chunk, ctot[c] = the chunk's weight; gram_assign_kernel adds the chunks before.
constexpr int GRAM_CHUNK = 4096;
constexpr int GRAM_MAX_CHUNKS = GRAM_MAX_G / GRAM_CHUNK;
__global__ void __launch_bounds__(1024)
gram_scan_kernel(const uint32_t *__restrict__ gh, uint32_t G, uint64_t smooth, uint64_t *__restrict__ cum,
                 uint64_t *__restrict__ ctot)
{
    const uint32_t tid = threadIdx.x;
    const uint32_t g0 = blockIdx.x * GRAM_CHUNK + tid * 4u;
    uint64_t w[4] = {0, 0, 0, 0};
    if (g0 + 4 <= G && (G & 3u) == 0) {
        const uint4 v = *reinterpret_cast<const uint4 *>(gh + g0);
        w[0] = 16ull * v.x + smooth; w[1] = 16ull * v.y + smooth; w[2] = 16ull * v.z + smooth; w[3] = 16ull * v.w + smooth;
    } else {
        for (int q = 0; q < 4; ++q) if (g0 + q < G) w[q] = 16ull * gh[g0 + q] + smooth;
    }
    uint64_t total;
    uint64_t run = block_excl_scan(w[0] + w[1] + w[2] + w[3], (uint64_t)0, Plus(), total);
    for (int q = 0; q < 4; ++q) {
        if (g0 + q < G) cum[g0 + q] = run;
        run += w[q];
    }
    if (tid == 0) ctot[blockIdx.x] = total;
}

// every leaf walks down from the root: a node [lo, hi) splits where its two halves weigh most alike (binary search on
// cum); left = 0, right = 1.  All leaves of a node compute the same split, so the codes are prefix-free and ordered.
__global__ void __launch_bounds__(64)
gram_assign_kernel(const uint64_t *__restrict__ cum, const uint64_t *__restrict__ ctot, const uint32_t *__restrict__ gh,
                   uint32_t G, uint32_t B, double samples, uint32_t *__restrict__ tab, double *__restrict__ stats)
{
    __shared__ uint64_t s_off[GRAM_MAX_CHUNKS + 1];
    const uint32_t nchunks = (G + GRAM_CHUNK - 1) / GRAM_CHUNK;
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (uint32_t c = 0; c < nchunks; ++c) { s_off[c] = run; run += ctot[c]; }
        s_off[nchunks] = run;
    }
    __syncthreads();
    // global exclusive prefix at x (x == G: the total weight)
    auto cumv = [&](uint32_t x) -> uint64_t { return x >= G ? s_off[nchunks] : cum[x] + s_off[x / GRAM_CHUNK]; };
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t len = 0, code = 0;
    bool ok = true;
    if (g < G) {
        uint32_t lo = 0, hi = G;
        uint64_t clo = 0, chi = cumv(G);
        while (hi - lo > 1) {
            const uint64_t target = clo + chi;                  // twice the midpoint weight
            uint32_t a = lo + 1, b = hi - 1;                     // smallest sp in [lo + 1, hi - 1] with 2 cum[sp] >= target
            while (a < b) {
                const uint32_t mid = a + ((b - a) >> 1);
                if (2 * cumv(mid) >= target) b = mid; else a = mid + 1;
            }
            uint32_t sp = a;
            uint64_t csp = cumv(sp);
            if (sp > lo + 1) {
                const uint64_t cpr = cumv(sp - 1);                // 2 cum[sp - 1] < target
                const uint64_t hi_d = 2 * csp >= target ? 2 * csp - target : target - 2 * csp;
                const uint64_t lo_d = target - 2 * cpr;
                if (lo_d <= hi_d) { sp = sp - 1; csp = cpr; }
            }
            if (g < sp) { hi = sp; chi = csp; code <<= 1; }
            else { lo = sp; clo = csp; code = (code << 1) | 1u; }
            if (++len > (uint32_t)GRAM_MAX_LEN) { ok = false; break; }
        }
        if (len == 0) len = 1;                                  // a single leaf (G == 1)
        tab[g] = ok ? ((code << (32 - len)) | len) : 0u;        // code word left-aligned above the 5 length bits
    }
    // statistics over the sample: code bits, longest code word, failures, mean and second moment of the information
    const double c = (g < G) ? (double)gh[g] : 0.0;
    double wl = ok ? c * len : 0.0, i1 = 0.0, i2 = 0.0, c1 = 0.0, c2 = 0.0;
    if (c > 0.0) {
        const double lp = log2(samples / c);
        i1 = c * lp;
        i2 = c * lp * lp;
        // the grams sharing this one's first k - 1 digits are the B consecutive table entries around it
        const uint32_t first = g - g % B;
        double cp = 0.0;
        for (uint32_t q = 0; q < B; ++q) cp += (double)gh[first + q];
        const double lc = log2(cp / c);
        c1 = c * lc;
        c2 = c * lc * lc;
    }
    for (int o = 16; o > 0; o >>= 1) {
        wl += __shfl_down_sync(0xffffffffu, wl, o);
        i1 += __shfl_down_sync(0xffffffffu, i1, o);
        i2 += __shfl_down_sync(0xffffffffu, i2, o);
        c1 += __shfl_down_sync(0xffffffffu, c1, o);
        c2 += __shfl_down_sync(0xffffffffu, c2, o);
    }
    uint32_t ml = (g < G) ? len : 0u;
    ml = __reduce_max_sync(0xffffffffu, ml);
    const uint32_t bad = __popc(__ballot_sync(0xffffffffu, g < G && !ok));
    if ((threadIdx.x & 31u) == 0) {
        if (wl > 0.0) atomicAdd(&stats[1], wl);
        if (i1 > 0.0) { atomicAdd(&stats[4], i1); atomicAdd(&stats[5], i2); }
        if (c1 > 0.0) { atomicAdd(&stats[6], c1); atomicAdd(&stats[7], c2); }
        // max over non-negative doubles through their bit patterns
        atomicMax(reinterpret_cast<unsigned long long *>(&stats[2]), (unsigned long long)__double_as_longlong((double)ml));
        if (bad) atomicAdd(&stats[3], (double)bad);
    }
}

int plan_round0(const uint64_t *h_hist, Round0Plan &p, const uint8_t *d_text, uint64_t n, const GramScratch *gs,
                cudaStream_t st)
{
    const char *e_bits0 = getenv("HKCSA_BITS0");       // tuning knob: the key width
    const char *e_gram = getenv("HKCSA_GRAM");
    const int want_bits0 = e_bits0 ? 8 * (atoi(e_bits0) / 8) : 0;
    uint32_t sigma = 0;
    for (int ch = 0; ch < 256; ++ch)
        if (h_hist[ch]) ++sigma;
    const int b = std::max(1, (int)bits_for(sigma));   // fixed-width code size, for reference
    // round-0 keys: the first bits0 bits of the alphabetic code stream; as many symbols on average as a
    // fixed-width packing of 64 / b symbols would hold, in fewer bits when the symbol distribution allows
    AlphaCode &ac = p.ac;
    double avg_len = b;
    int max_len = b;
    if (!build_alpha_code(h_hist, ac, avg_len, max_len)) {
        uint32_t code = 0;                               // degenerate distribution: fixed-width codes
        ac.code[256] = 0; ac.len[256] = (uint8_t)b;
        for (int ch = 0; ch < 256; ++ch)
            if (h_hist[ch]) { ac.code[ch] = ++code; ac.len[ch] = (uint8_t)b; }
        avg_len = max_len = b;
    }
    const int k_target = 64 / b;
    int bits0 = 8 * (int)ceil(k_target * avg_len / 8.0 - 1e-9);
    bits0 = std::max(16, std::min(64, bits0));
    if (e_bits0) bits0 = std::max(16, std::min(64, want_bits0));
    p.sigma = sigma;
    p.b = b;
    p.max_len = max_len;
    p.bits0 = bits0;
    p.k0 = std::max(1, bits0 / max_len);         // symbols every key is guaranteed to cover
    p.passes0 = bits0 / 8;

    // ---- the k-gram code (suffix_array.cuh): sampled gram histogram -> code built on the device -> its statistics
    //      decide the key width.  Small texts and failures keep the per-symbol code above.
    GramCode &gc = p.gram;
    gc.tab = nullptr;
    const uint32_t B = sigma + 1;
    uint32_t k = 1, G = B;
    while (k < (uint32_t)GRAM_MAX_K && (uint64_t)G * B <= (uint64_t)GRAM_MAX_G) { G *= B; ++k; }
    if (!d_text || n < 1024 || k < (uint32_t)GRAM_MIN_K || (e_gram && atoi(e_gram) == 0)) return HKCSA_OK;
    memset(gc.digit, 0, sizeof(gc.digit));
    uint32_t dgt = 0;
    for (int ch = 0; ch < 256; ++ch)
        if (h_hist[ch]) gc.digit[ch] = (uint8_t)++dgt;      // k >= 4 means B <= 19
    gc.k = k; gc.B = B; gc.G = G;
    gc.pw = 1;
    for (uint32_t q = 1; q < k; ++q) gc.pw *= B;
    const uint32_t N = (uint32_t)n;
    const uint32_t tiles = (N + PACK_TILE - 1) / PACK_TILE;
    const uint32_t stride = std::max<uint32_t>(1, tiles / 256);           // about half a million samples at most
    uint8_t *pin = static_cast<uint8_t *>(pinned_page());
    HK_REQUIRE(pin != nullptr, HKCSA_ECUDA, "pinned page allocation failed");
    double *h_gs = reinterpret_cast<double *>(pin + 2560);
    HK_CUDA(cudaMemsetAsync(gs->hist, 0, (size_t)G * sizeof(uint32_t), st));
    HK_CUDA(cudaMemsetAsync(gs->stats, 0, 8 * sizeof(uint64_t), st));
    // the sampled positions: every stride-th tile of 2048
    uint64_t nsamp = 0;
    for (uint32_t t = 0; t < tiles; t += stride) nsamp += std::min<uint64_t>(PACK_TILE, n - (uint64_t)t * PACK_TILE);
    const uint64_t smooth = std::max<uint64_t>(1, nsamp / G);
    uint64_t *d_ctot = gs->cum + GRAM_MAX_G + 8;
    {
        prof::Scope ps(st, prof::OTHER, (uint64_t)N / stride + (uint64_t)G * 24);
        gram_hist_kernel<<<(tiles + stride - 1) / stride, PACK_THREADS, 0, st>>>(d_text, N, gc, stride, gs->hist);
        HK_LAUNCH_CHECK();
        gram_scan_kernel<<<(G + GRAM_CHUNK - 1) / GRAM_CHUNK, 1024, 0, st>>>(gs->hist, G, smooth, gs->cum, d_ctot);
        HK_LAUNCH_CHECK();
        gram_assign_kernel<<<(G + 63) / 64, 64, 0, st>>>(gs->cum, d_ctot, gs->hist, G, B, (double)nsamp, gs->tab,
                                                         reinterpret_cast<double *>(gs->stats));
        HK_LAUNCH_CHECK();
    }
    HK_CUDA(cudaMemcpyAsync(h_gs, gs->stats, 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    if (!(nsamp > 0 && h_gs[3] == 0 && h_gs[2] >= 1 && h_gs[2] <= (double)GRAM_MAX_LEN)) return HKCSA_OK;
    gc.tab = gs->tab;
    const double samples = (double)nsamp;
    const double gram_len = h_gs[1] / samples;                          // mean code bits per gram
    const double mu = h_gs[4] / samples;                                // information per gram: mean ...
    const double var = std::max(1e-9, h_gs[5] / samples - mu * mu);     // ... and variance
    const int gram_max_len = (int)h_gs[2];
    const int min_bits = std::max(16, 8 * ((gram_max_len + 7) / 8));    // a key holds at least one whole gram
    const double h_rate = h_gs[6] / samples;                            // information of a symbol given the k - 1 before it
    const double h_var = std::max(1e-9, h_gs[7] / samples - h_rate * h_rate);
    // Key width: the narrowest whose predicted survivors stay under 0.5 % of the suffixes.  A key of `cand` code bits
    // covers s = cand * k / gram_len symbols; their information is about normal with the first gram's marginal mean /
    // variance plus, per further symbol, the conditional ones (the text's entropy rate at order k - 1: the marginal
    // statistics of DNA 6-grams are nearly flat, the skew sits in the conditionals).  A suffix survives round 0 when
    // its key is likelier than 1 / n.  A survivor costs about as much as 40 elements of a radix pass, so a pass is
    // worth dropping while it adds less than 2.5 % survivors; the prediction ran 4x low on the DNA workload, hence 0.5 %.
    int bits = 64;
    for (int cand = min_bits; cand <= 64; cand += 8) {
        const double more = std::max(0.0, cand * (double)k / gram_len - k);
        const double z = (log2((double)n) - (mu + more * h_rate)) / sqrt(var + more * h_var);
        if (0.5 * erfc(-z / sqrt(2.0)) <= 0.005) { bits = cand; break; }
    }
    if (getenv("HKCSA_DEBUG_PLAN"))
        fprintf(stderr, "[hkcsa] gram code: k=%u B=%u G=%u samples=%.0f len/gram=%.3f max_len=%d info/gram=%.3f var=%.3f "
                "rate=%.3f var=%.3f -> bits0=%d\n", k, B, G, samples, gram_len, gram_max_len, mu, var, h_rate, h_var, bits);
    if (e_bits0) bits = std::max(min_bits, std::min(64, want_bits0));
    p.bits0 = bits;
    p.max_len = gram_max_len;
    p.k0 = (int)k * std::max(1, std::min(GRAM_PER_KEY, bits / gram_max_len));
    p.passes0 = bits / 8;
    return HKCSA_OK;
}

// ---------------------------------------------------------------- round 0: pack
// key[i] = the first 8 * PASSES bits of the code stream of suffix i, from the key source Keys (suffix_array.cuh).
// Keys are produced warp-striped so the stores are fully coalesced.  The suffix ids are not written at all: the first
// radix pass takes "value = index" (radix_sort_pairs_u64, identity_vals).
// PASSES = radix passes of round 0 = key bits / 8, a template parameter: the key shift and the digit histogram of
// every pass (the bulk of the kernel's instructions: one shared atomic per key and pass) are straight-line code.
// CARRY: the symbol before the suffix (its BWT symbol, csa/bwt.py:6-11) rides in the top byte of the key, above
// the sorted bits (keys of at most 56 bits): the sort delivers the BWT in suffix-array order and nobody has to gather
// text[SA[i] - 1] at random afterwards.
// Persistent: a CTA takes every gridDim.x-th tile, so the digit histograms leave shared memory once per CTA, not once
// per tile (1536 global atomics per 2048 keys otherwise: 0.55 -> 0.48 ms at C2), and the code tables are set up once.
template <typename Keys, int PASSES, bool CARRY>
__global__ void __launch_bounds__(PACK_THREADS, 6)
sa_pack0_kernel(const uint8_t *__restrict__ text, uint32_t n, Keys src, uint64_t *__restrict__ keys,
                uint32_t *__restrict__ ghist)
{
    static_assert(!CARRY || PASSES <= 7, "the carried symbol needs the top byte of the key");
    constexpr int bits = 8 * PASSES;
    __shared__ typename Keys::Smem s;
    __shared__ uint32_t s_hist[8 * RADIX];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    hist_zero(s_hist, PASSES);
    src.setup(s);
    __syncthreads();
    const bool aligned8 = (reinterpret_cast<uintptr_t>(text) & 7) == 0;
    const uint32_t tiles = (n + PACK_TILE - 1) / PACK_TILE;
    for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const uint64_t base = (uint64_t)tile * PACK_TILE;
        src.fill(s, text, n, base, aligned8);
#pragma unroll
        for (int e = 0; e < PACK_IPT; ++e) {
            const uint32_t j = warp * (32u * PACK_IPT) + e * 32u + lane;
            const uint64_t g = base + j;
            const uint64_t key = src.window(s, j, bits) >> (64 - bits);
            const bool valid = g < n;
            if (valid) {
                if (CARRY) keys[g] = key | ((uint64_t)__ldg(text + (g ? g - 1 : (uint64_t)n - 1)) << 56);   // an L1 hit: the tile was just read
                else keys[g] = key;
            }
            hist_add_key_unsorted<PASSES>(s_hist, key, valid);
        }
        __syncthreads();      // the next tile overwrites the tile storage
    }
    hist_flush(s_hist, ghist, PASSES);
}

// sa_pack0_kernel<Keys, passes, carry> over the whole text (carry needs passes <= 7)
template <typename Keys, int P = 2>
static void launch_pack0(const Keys &src, int passes, bool carry, const uint8_t *text, uint32_t n, uint64_t *keys,
                         uint32_t *ghist, cudaStream_t st)
{
    if constexpr (P < 8) {
        if (passes != P) return launch_pack0<Keys, P + 1>(src, passes, carry, text, n, keys, ghist, st);
    }
    const uint32_t blocks = std::min<uint32_t>((n + PACK_TILE - 1) / PACK_TILE, (uint32_t)num_sms() * 6u);
    if constexpr (P < 8) {
        if (carry) { sa_pack0_kernel<Keys, P, true><<<blocks, PACK_THREADS, 0, st>>>(text, n, src, keys, ghist); return; }
    }
    sa_pack0_kernel<Keys, P, false><<<blocks, PACK_THREADS, 0, st>>>(text, n, src, keys, ghist);
}

// ---------------------------------------------------------------- later rounds: key build
// key[j] = (group start << b2) | (rank(idx + h) + 1), low part 0 when idx + h >= n.
//
// rank(t) comes from the rank array when it was scattered for every suffix (EAGER), or -- when only a
// small fraction of the suffixes survived round 0 (LAZY) -- is recomputed on demand: a suffix that was
// already unique after round 0 has rank = lower_bound of its round-0 key in the sorted round-0 keys, so
// the 4-byte random scatter of n ranks is replaced by a binary search for the few ranks that are read.
// Suffixes that were NOT unique after round 0 always have their current rank in the array.
struct LazyRank {
    const uint8_t *text;       // nullptr = eager mode
    const uint64_t *keys0;     // round-0 keys, sorted
    const uint32_t *bucket;    // bucket[v] = lower_bound(keys0, v << shift), v in [0, 2^bucket_bits]
    const uint64_t *samples;   // samples[j] = keys0[j << LAZY_SAMPLE_SHIFT]
    int first_round;           // round 1: every rank still IS the round-0 group start = the lower bound itself,
                               // so the rank array is neither written in round 0 nor read here
    int bits;                  // width of a round-0 key
    int shift;                 // key >> shift = bucket id
    uint64_t mask;             // the sorted bits of a round-0 key (the top byte may carry the BWT symbol)
    GramKeys gram;             // gram.code.tab != nullptr: round-0 keys come from the k-gram code
};

constexpr int LAZY_BUCKET_BITS = 20;
// Every 64th sorted key, kept apart: n / 8 bytes (25 MB at C3), L2-resident, so the long part of a look-up's
// binary search (buckets of frequent prefixes hold millions of keys) runs on L2 hits and only the last six
// steps -- inside 64 consecutive keys = four lines -- go to DRAM.
constexpr int LAZY_SAMPLE_SHIFT = 6;

__global__ void sa_key_samples_kernel(const uint64_t *__restrict__ keys0, uint32_t n, uint64_t mask,
                                      uint64_t *__restrict__ samples)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (((uint64_t)j << LAZY_SAMPLE_SHIFT) < n) samples[j] = keys0[(uint64_t)j << LAZY_SAMPLE_SHIFT] & mask;
}

// bucket[v] = lower_bound(keys0, v << shift) for v in [0, nbuckets]: one binary search per bucket
// boundary (2^20 searches whose upper levels stay in L2), not a pass over the keys
__global__ void sa_bucket_index_kernel(const uint64_t *__restrict__ keys0, uint32_t n, int shift, uint64_t mask,
                                       uint32_t nbuckets, uint32_t *__restrict__ bucket)
{
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v > nbuckets) return;
    uint32_t lo = 0, hi = n;
    if (v == nbuckets) lo = n;
    const uint64_t key = (uint64_t)v << shift;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if ((__ldg(keys0 + mid) & mask) < key) lo = mid + 1; else hi = mid;
    }
    bucket[v] = lo;
}

// COHERENT: the rank array is written by the calling kernel itself (sa_finish_small_kernel): read it with volatile loads
template <bool COHERENT = false>
__device__ __forceinline__ uint32_t lazy_rank_lookup(const LazyRank &lz, const AlphaKeys::Tab &s_tab, uint32_t n,
                                                     uint32_t t, const uint32_t *rank)
{
    const uint64_t key = lz.gram.code.tab ? lz.gram.at(lz.text, n, t, lz.bits) : AlphaKeys::at(s_tab, lz.text, n, t, lz.bits);
    const uint32_t v = (uint32_t)(key >> lz.shift);
    uint32_t lo = __ldg(lz.bucket + v), hi = __ldg(lz.bucket + v + 1);
    if (hi - lo > (2u << LAZY_SAMPLE_SHIFT)) {
        // first the samples whose positions lie in [lo, hi): smallest j with samples[j] >= key
        const uint32_t jlo = (lo + (1u << LAZY_SAMPLE_SHIFT) - 1u) >> LAZY_SAMPLE_SHIFT;
        const uint32_t jhi = (hi + (1u << LAZY_SAMPLE_SHIFT) - 1u) >> LAZY_SAMPLE_SHIFT;
        uint32_t a = jlo, b = jhi;
        while (a < b) {
            const uint32_t mid = a + ((b - a) >> 1);
            if (__ldg(lz.samples + mid) < key) a = mid + 1; else b = mid;
        }
        // the answer lies in (position of sample a-1, position of sample a], clipped to [lo, hi)
        if (a > jlo) lo = max(lo, ((a - 1u) << LAZY_SAMPLE_SHIFT) + 1u);
        if (a < jhi) hi = min(hi, a << LAZY_SAMPLE_SHIFT);
    }
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if ((__ldg(lz.keys0 + mid) & lz.mask) < key) lo = mid + 1; else hi = mid;
    }
    if (lz.first_round) return lo;
    const bool shared_group = (lo + 1 < n) && ((__ldg(lz.keys0 + lo + 1) & lz.mask) == key);
    if (!shared_group) return lo;
    return COHERENT ? *reinterpret_cast<const volatile uint32_t *>(rank + t) : rank[t];
}

__global__ void __launch_bounds__(256)
sa_keybuild_kernel(const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp,
                   const uint32_t *__restrict__ rank, uint32_t n, uint32_t h, int b2, uint32_t m, int passes,
                   uint64_t *__restrict__ keys, uint32_t *__restrict__ ghist, LazyRank lz, AlphaCode ac)
{
    __shared__ uint32_t s_hist[8 * RADIX];
    __shared__ AlphaKeys::Tab s_tab;
    s_tab.load(ac);
    hist_zero(s_hist, passes);
    __syncthreads();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < m; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t j = base + threadIdx.x;
        const bool valid = j < m;
        uint64_t key = 0;
        if (valid) {
            const uint32_t i = cidx[j];
            const uint64_t t = (uint64_t)i + h;
            uint32_t k2 = 0;
            if (t < n) k2 = (lz.text ? lazy_rank_lookup(lz, s_tab, n, (uint32_t)t, rank) : rank[t]) + 1u;
            key = ((uint64_t)cgrp[j] << b2) | k2;
            keys[j] = key;
        }
        hist_add_key(s_hist, key, passes, valid);
    }
    __syncthreads();
    hist_flush(s_hist, ghist, passes);
}

// ---------------------------------------------------------------- segmented rank update
// After a sort, over the m working elements (sorted keys skey, suffix ids sidx,
// SA slots pos -- identity in round 0):
//   head[j]   = j == 0 || skey[j] != skey[j-1]
//   single[j] = head[j] && (j == m-1 || head[j+1])
//   grp[j]    = pos[last head <= j]            (max-scan)
//   SA[pos[j]] = sidx[j];  rank[sidx[j]] = grp[j]
//   non-singletons are compacted into (cpos, cidx, cgrp) for the next round.
// Three phases (tile reduce, scan of tile aggregates, apply) -- no spinning.

// `mask` = the key bits that were sorted on; *carried = the top bytes of the thread's eight keys, first key lowest
__device__ __forceinline__ void seg_flags(const uint64_t *__restrict__ skey, uint32_t m, uint32_t j0, uint64_t mask,
                                          bool head[SEG_IPT], bool single[SEG_IPT], uint64_t *carried)
{
    // thread owns j0 .. j0+SEG_IPT-1 (blocked): four 16-byte loads; the keys just outside (j0-1 and
    // j0+SEG_IPT) come from the neighbouring lanes, only the warp's two edge lanes load them.
    // Must be called by all 32 lanes of the warp.
    uint64_t k[SEG_IPT + 2];
    if (j0 + SEG_IPT <= m) {
        const ulonglong2 *v = reinterpret_cast<const ulonglong2 *>(skey + j0);   // j0 is a multiple of 8: 64-byte aligned
#pragma unroll
        for (int e = 0; e < SEG_IPT / 2; ++e) {
            const ulonglong2 q = v[e];
            k[1 + 2 * e] = q.x;
            k[2 + 2 * e] = q.y;
        }
    } else {
#pragma unroll
        for (int e = 0; e < SEG_IPT; ++e) k[1 + e] = (j0 + e < m) ? skey[j0 + e] : 0ULL;
    }
    const uint32_t lane = lane_id();
    uint64_t prev = __shfl_up_sync(0xffffffffu, k[SEG_IPT], 1);
    uint64_t next = __shfl_down_sync(0xffffffffu, k[1], 1);
    if (lane == 0) prev = (j0 > 0 && j0 - 1 < m) ? skey[j0 - 1] : 0ULL;
    if (lane == 31) next = (j0 + SEG_IPT < m) ? skey[j0 + SEG_IPT] : 0ULL;
    k[0] = prev;
    k[SEG_IPT + 1] = next;
    if (carried) {
        uint64_t c = 0;
#pragma unroll
        for (int e = 0; e < SEG_IPT; ++e) c |= (k[1 + e] >> 56) << (8 * e);
        *carried = c;
    }
#pragma unroll
    for (int e = 0; e < SEG_IPT + 2; ++e) k[e] &= mask;
#pragma unroll
    for (int e = 0; e < SEG_IPT; ++e) {
        const uint32_t j = j0 + e;
        const bool in = j < m;
        const bool hd = in && (j == 0 || k[e + 1] != k[e]);
        const bool next_head = (j + 1 >= m) || (k[e + 2] != k[e + 1]);
        head[e] = hd;
        single[e] = hd && next_head;
    }
}

__global__ void __launch_bounds__(SEG_THREADS)
seg_reduce_kernel(const uint64_t *__restrict__ skey, uint32_t m, uint32_t *__restrict__ agg_head,
                  uint32_t *__restrict__ agg_keep, uint16_t *__restrict__ flags, uint64_t mask,
                  uint8_t *__restrict__ carried_out)
{
    __shared__ uint32_t s_h[SEG_THREADS / 32], s_k[SEG_THREADS / 32];
    const uint32_t tid = threadIdx.x;
    const uint32_t j0 = blockIdx.x * SEG_TILE + tid * SEG_IPT;
    bool head[SEG_IPT], single[SEG_IPT];
    uint64_t carried = 0;
    seg_flags(skey, m, j0, mask, head, single, carried_out ? &carried : nullptr);
    if (carried_out) {
        // round 0 with the BWT symbol in the top byte of the key: row j of the BWT is the top byte of sorted key j
        // (rows of suffixes that are not yet in their final slot are written again by the round that places them)
        if (j0 + SEG_IPT <= m && (reinterpret_cast<uintptr_t>(carried_out) & 7) == 0) {
            *reinterpret_cast<uint64_t *>(carried_out + j0) = carried;
        } else {
            for (int e = 0; e < SEG_IPT && j0 + e < m; ++e) carried_out[j0 + e] = (uint8_t)(carried >> (8 * e));
        }
    }
    uint32_t lasthead = 0, keep = 0;   // lasthead = (index of last head) + 1, 0 = none
    uint32_t f = 0;
#pragma unroll
    for (int e = 0; e < SEG_IPT; ++e) {
        if (head[e]) lasthead = j0 + e + 1;
        if (j0 + e < m && !single[e]) ++keep;
        f |= (head[e] ? 1u : 0u) << e;
        f |= (single[e] ? 1u : 0u) << (SEG_IPT + e);
    }
    // 2 bits per element for the apply pass: it then reads 0.25 B instead of the 8-byte key again
    flags[blockIdx.x * SEG_THREADS + tid] = (uint16_t)f;
    lasthead = __reduce_max_sync(0xffffffffu, lasthead);
    keep = __reduce_add_sync(0xffffffffu, keep);
    if ((tid & 31u) == 0) { s_h[tid >> 5] = lasthead; s_k[tid >> 5] = keep; }
    __syncthreads();
    if (tid == 0) {
        uint32_t h = 0, k = 0;
        for (int w = 0; w < SEG_THREADS / 32; ++w) { h = max(h, s_h[w]); k += s_k[w]; }
        agg_head[blockIdx.x] = h;
        agg_keep[blockIdx.x] = k;
    }
}

// single CTA: exclusive (max, sum) scan over tile aggregates, in place; total keep -> *out_m.
// Two levels: warp w owns a contiguous range of the tiles, reduces it, and the 32 warp totals give every warp its carry;
// then each warp scans its range in steps of 32 lanes x SCAN_IPT tiles (16-byte loads), loading the next step before
// it stores the current one.  (The one-level form went through the tiles 4096 at a time with four barriers and a
// serial pass over the warp totals per step: 37 us for the 48.8 k tiles of C2.)
constexpr int SCAN_IPT = 8;
constexpr uint32_t SCAN_STEP = 32 * SCAN_IPT;      // tiles a warp scans per step

struct ScanStep {
    uint32_t h[SCAN_IPT], k[SCAN_IPT];
};

// tiles [i, i + SCAN_IPT) of the two arrays, zeros from `end` on (i is a multiple of 8: 32-byte aligned)
__device__ __forceinline__ void scan_load(const uint32_t *agg_head, const uint32_t *agg_keep, uint32_t i, uint32_t end,
                                          ScanStep &v)
{
    if (i + SCAN_IPT <= end) {
#pragma unroll
        for (int q = 0; q < SCAN_IPT; q += 4) {
            const uint4 a = *reinterpret_cast<const uint4 *>(agg_head + i + q);
            const uint4 b = *reinterpret_cast<const uint4 *>(agg_keep + i + q);
            v.h[q] = a.x; v.h[q + 1] = a.y; v.h[q + 2] = a.z; v.h[q + 3] = a.w;
            v.k[q] = b.x; v.k[q + 1] = b.y; v.k[q + 2] = b.z; v.k[q + 3] = b.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < SCAN_IPT; ++q) {
            v.h[q] = i + q < end ? agg_head[i + q] : 0u;
            v.k[q] = i + q < end ? agg_keep[i + q] : 0u;
        }
    }
}

__global__ void __launch_bounds__(1024)
seg_scan_kernel(uint32_t *__restrict__ agg_head, uint32_t *__restrict__ agg_keep, uint32_t tiles,
                uint32_t *__restrict__ out_m)
{
    __shared__ uint32_t s_h[32], s_k[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t per = (tiles + 32 * SCAN_STEP - 1) / (32 * SCAN_STEP) * SCAN_STEP;
    const uint32_t lo = min(warp * per, tiles), hi = min(lo + per, tiles);
    // level 1: (max, sum) of the warp's range -- independent loads
    uint32_t th = 0, tk = 0;
#pragma unroll 2
    for (uint32_t i = lo + lane * SCAN_IPT; i < hi; i += SCAN_STEP) {
        ScanStep v;
        scan_load(agg_head, agg_keep, i, hi, v);
#pragma unroll
        for (int q = 0; q < SCAN_IPT; ++q) { th = max(th, v.h[q]); tk += v.k[q]; }
    }
    th = __reduce_max_sync(0xffffffffu, th);
    tk = __reduce_add_sync(0xffffffffu, tk);
    if (lane == 0) { s_h[warp] = th; s_k[warp] = tk; }
    __syncthreads();
    uint32_t ch = __reduce_max_sync(0xffffffffu, lane < warp ? s_h[lane] : 0u);     // carry into this warp's range
    uint32_t ck = __reduce_add_sync(0xffffffffu, lane < warp ? s_k[lane] : 0u);
    const uint32_t total = __reduce_add_sync(0xffffffffu, s_k[lane]);
    if (tid == 0) *out_m = total;
    // level 2: the warp's range, one step of 32 x SCAN_IPT tiles after the other
    ScanStep cur;
    if (lo < hi) scan_load(agg_head, agg_keep, lo + lane * SCAN_IPT, hi, cur);
    for (uint32_t i = lo; i < hi; i += SCAN_STEP) {
        ScanStep nxt;
        if (i + SCAN_STEP < hi) scan_load(agg_head, agg_keep, i + SCAN_STEP + lane * SCAN_IPT, hi, nxt);
        uint32_t lh = 0, lk = 0;
#pragma unroll
        for (int q = 0; q < SCAN_IPT; ++q) { lh = max(lh, cur.h[q]); lk += cur.k[q]; }
        const uint32_t ih = warp_incl_max(lh);
        uint32_t step_k;
        const uint32_t ek = warp_excl_sum(lk, step_k);
        const uint32_t up = __shfl_up_sync(0xffffffffu, ih, 1);
        uint32_t run_h = max(ch, lane ? up : 0u), run_k = ck + ek;
        const uint32_t x = i + lane * SCAN_IPT;
#pragma unroll
        for (int q = 0; q < SCAN_IPT; ++q) {
            const uint32_t h = cur.h[q], k = cur.k[q];
            cur.h[q] = run_h;
            cur.k[q] = run_k;
            run_h = max(run_h, h);
            run_k += k;
        }
        if (x + SCAN_IPT <= hi) {
#pragma unroll
            for (int q = 0; q < SCAN_IPT; q += 4) {
                *reinterpret_cast<uint4 *>(agg_head + x + q) = make_uint4(cur.h[q], cur.h[q + 1], cur.h[q + 2], cur.h[q + 3]);
                *reinterpret_cast<uint4 *>(agg_keep + x + q) = make_uint4(cur.k[q], cur.k[q + 1], cur.k[q + 2], cur.k[q + 3]);
            }
        } else {
#pragma unroll
            for (int q = 0; q < SCAN_IPT; ++q)
                if (x + q < hi) { agg_head[x + q] = cur.h[q]; agg_keep[x + q] = cur.k[q]; }
        }
        ch = max(ch, __shfl_sync(0xffffffffu, ih, 31));
        ck += step_k;
        cur = nxt;
    }
}

// Rounds that place suffixes (write_sa), and round 0 with ranks for every suffix (scatter_all): per element the SA slot,
// the suffix id, the rank scatter and -- for survivors -- the compacted triple.  A thread's eight ids and slots come in
// with 16-byte loads and its eight BWT symbols are read before anything is stored, so the random reads of a thread
// are in flight together.
__global__ void __launch_bounds__(SEG_THREADS, 6)
seg_apply_kernel(const uint16_t *__restrict__ flags, const uint32_t *__restrict__ sidx,
                 const uint32_t *__restrict__ pos /* nullptr = identity */, uint32_t m,
                 const uint32_t *__restrict__ carry_head, const uint32_t *__restrict__ carry_keep,
                 uint32_t *__restrict__ sa, uint32_t *__restrict__ rank, uint32_t *__restrict__ cpos,
                 uint32_t *__restrict__ cidx, uint32_t *__restrict__ cgrp, bool write_sa, bool scatter_all,
                 const uint8_t *__restrict__ text, uint32_t n, uint8_t *__restrict__ bwt)
{
    __shared__ uint32_t s_h[SEG_THREADS / 32], s_k[SEG_THREADS / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t j0 = blockIdx.x * SEG_TILE + tid * SEG_IPT;
    const uint32_t f = flags[blockIdx.x * SEG_THREADS + tid];      // written by seg_reduce_kernel
    // last head and survivors of this thread's eight elements straight from the flag bits
    const uint32_t h8 = f & 0xFFu, s8 = (f >> SEG_IPT) & 0xFFu;
    const uint32_t vm = (j0 + SEG_IPT <= m) ? 0xFFu : (j0 < m ? (1u << (m - j0)) - 1u : 0u);
    const uint32_t lasthead = h8 ? j0 + (32u - __clz(h8)) : 0u;
    const uint32_t keep = __popc(~s8 & vm);
    // block-wide exclusive (max, sum) scan over threads.  The last-head values grow with the lane, so the running
    // maximum before a lane is the value of the nearest lower lane that has a head: one ballot and one shuffle; the
    // survivor counts (<= 8) are summed bit by bit with four ballots.
    const uint32_t lt = lanemask_lt();
    const uint32_t hb = __ballot_sync(0xffffffffu, h8 != 0u);
    const uint32_t lower = hb & lt;
    uint32_t eh = __shfl_sync(0xffffffffu, lasthead, lower ? 31 - __clz(lower) : 0);
    if (!lower) eh = 0;
    uint32_t ek = 0, wk_total = 0;
#pragma unroll
    for (int bit = 0; bit < 4; ++bit) {
        const uint32_t kb = __ballot_sync(0xffffffffu, (keep >> bit) & 1u);
        ek += (uint32_t)__popc(kb & lt) << bit;
        wk_total += (uint32_t)__popc(kb) << bit;
    }
    const uint32_t wh = __shfl_sync(0xffffffffu, lasthead, hb ? 31 - __clz(hb) : 0);     // the warp's last head
    if (lane == 31) { s_h[warp] = hb ? wh : 0u; s_k[warp] = wk_total; }
    __syncthreads();
    if (!vm) return;
    uint32_t ph = carry_head[blockIdx.x], pk = carry_keep[blockIdx.x];
    for (uint32_t w = 0; w < warp; ++w) { ph = max(ph, s_h[w]); pk += s_k[w]; }
    const uint32_t head_in = max(ph, eh);   // (index of the governing head) + 1 before this thread's first element
    uint32_t s[SEG_IPT], p[SEG_IPT];
    if (vm == 0xFFu) {                      // j0 is a multiple of 8: 32-byte aligned
        const uint4 *vs = reinterpret_cast<const uint4 *>(sidx + j0);
        const uint4 a = vs[0], b = vs[1];
        s[0] = a.x; s[1] = a.y; s[2] = a.z; s[3] = a.w; s[4] = b.x; s[5] = b.y; s[6] = b.z; s[7] = b.w;
        if (pos) {
            const uint4 *vp = reinterpret_cast<const uint4 *>(pos + j0);
            const uint4 c = vp[0], d = vp[1];
            p[0] = c.x; p[1] = c.y; p[2] = c.z; p[3] = c.w; p[4] = d.x; p[5] = d.y; p[6] = d.z; p[7] = d.w;
        }
    } else {
#pragma unroll
        for (int e = 0; e < SEG_IPT; ++e) {
            s[e] = (vm >> e) & 1u ? sidx[j0 + e] : 0u;
            if (pos) p[e] = (vm >> e) & 1u ? pos[j0 + e] : 0u;
        }
    }
    if (!pos) {
#pragma unroll
        for (int e = 0; e < SEG_IPT; ++e) p[e] = j0 + e;
    }
    // group of the elements before this thread's first head: the slot of a head that lies in an earlier thread
    uint32_t grp = (h8 & 1u) ? 0u : (pos ? pos[head_in - 1] : head_in - 1);
    uint8_t c[SEG_IPT];
    if (write_sa && bwt) {                  // BWT rows carried by round 0: this slot's row follows its suffix
#pragma unroll
        for (int e = 0; e < SEG_IPT; ++e) c[e] = (vm >> e) & 1u ? text[s[e] ? s[e] - 1u : n - 1u] : 0;
    }
    uint32_t slot = pk + ek;
#pragma unroll
    for (int e = 0; e < SEG_IPT; ++e) {
        if (!((vm >> e) & 1u)) break;
        if ((h8 >> e) & 1u) grp = p[e];
        const bool single = (s8 >> e) & 1u;
        if (write_sa) {
            sa[p[e]] = s[e];
            if (bwt) bwt[p[e]] = c[e];
        }
        if (rank && (scatter_all || !single)) rank[s[e]] = grp;
        if (!single) {
            cpos[slot] = p[e];
            cidx[slot] = s[e];
            cgrp[slot] = grp;
            ++slot;
        }
    }
}

// Round 0 without rank scatter (lazy ranks; the distributed build's first refinement): only the survivors -- 0.3-3 %
// of the suffixes -- are written, compacted in order into (cpos, cidx, cgrp).  The flags are the whole input, so a CTA
// covers C0_TILES scan tiles, 64 elements per thread from one 16-byte flag load; its carry is the scanned aggregate of
// its first tile, and the prefix inside the CTA comes from the flag bits.  (One CTA per 2048-element tile made this a
// pass of 330 CTAs per SM, each waiting on two dependent loads to find nothing to do.)
constexpr int C0_THREADS = 512;
constexpr int C0_IPT = 64;
constexpr int C0_TILES = C0_THREADS * C0_IPT / SEG_TILE;
static_assert(C0_TILES * SEG_TILE == C0_THREADS * C0_IPT && C0_IPT == 8 * SEG_IPT, "a thread reads 8 flag words");

__global__ void __launch_bounds__(C0_THREADS, 3)
seg_compact0_kernel(const uint16_t *__restrict__ flags, const uint32_t *__restrict__ sidx, uint32_t m,
                    const uint32_t *__restrict__ carry_head, const uint32_t *__restrict__ carry_keep,
                    uint32_t *__restrict__ cpos, uint32_t *__restrict__ cidx, uint32_t *__restrict__ cgrp)
{
    __shared__ uint32_t s_h[C0_THREADS / 32], s_k[C0_THREADS / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t j0 = blockIdx.x * (uint32_t)(C0_THREADS * C0_IPT) + tid * C0_IPT;
    // the CTA's carry is loaded with its flags, not after the barrier: the pass is a chain of latencies per CTA
    const uint32_t t0 = blockIdx.x * (uint32_t)C0_TILES;
    const uint32_t carry_h = carry_head[t0], carry_k = carry_keep[t0];
    uint64_t hm = 0, sv = 0;                // head and survivor bits of elements j0 .. j0 + 63
    if (j0 < m) {
        const uint4 q = *reinterpret_cast<const uint4 *>(flags + (j0 >> 3));   // 8 flag words: bit e head, 8 + e singleton
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
        uint64_t single = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t f = w[i >> 1] >> (16 * (i & 1));
            hm |= (uint64_t)(f & 0xFFu) << (8 * i);
            single |= (uint64_t)((f >> 8) & 0xFFu) << (8 * i);
        }
        const uint64_t vm = (m - j0 >= (uint32_t)C0_IPT) ? ~0ull : (1ull << (m - j0)) - 1ull;
        sv = ~single & vm;
    }
    const uint32_t lasthead = hm ? j0 + 64u - (uint32_t)__clzll(hm) : 0u;      // (index of the last head) + 1
    const uint32_t ih = warp_incl_max(lasthead);
    uint32_t wk_total;
    const uint32_t ek = warp_excl_sum((uint32_t)__popcll(sv), wk_total);
    const uint32_t up = __shfl_up_sync(0xffffffffu, ih, 1);
    const uint32_t eh = lane ? up : 0u;
    if (lane == 31) { s_h[warp] = ih; s_k[warp] = wk_total; }
    __syncthreads();
    if (!sv) return;
    uint32_t ph = carry_h, pk = carry_k;
    for (uint32_t w = 0; w < warp; ++w) { ph = max(ph, s_h[w]); pk += s_k[w]; }
    const uint32_t head_in = max(ph, eh);
    uint32_t slot = pk + ek;
    // survivors cluster (repeats): a thread may hold 64 of them, so their ids are read eight at a time, the loads in
    // flight together -- one by one, each store waited for its load (57 us at C2, most of it in such threads)
    do {
        uint32_t e[8], id[8];
        int cnt = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            e[q] = sv ? (uint32_t)__ffsll((long long)sv) - 1u : 0u;
            if (sv) ++cnt;
            sv &= sv - 1ull;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) id[q] = q < cnt ? sidx[j0 + e[q]] : 0u;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (q >= cnt) break;
            const uint64_t hb = hm & (~0ull >> (63u - e[q]));                   // heads at or before element e
            cpos[slot] = j0 + e[q];
            cidx[slot] = id[q];
            cgrp[slot] = hb ? j0 + 63u - (uint32_t)__clzll(hb) : head_in - 1u;
            ++slot;
        }
    } while (sv);
}

void seg_compact0(const uint16_t *flags, const uint32_t *sidx, uint32_t m, const uint32_t *carry_head,
                  const uint32_t *carry_keep, uint32_t *cpos, uint32_t *cidx, uint32_t *cgrp, cudaStream_t st)
{
    const uint32_t blocks = (uint32_t)(((uint64_t)m + C0_THREADS * C0_IPT - 1) / (C0_THREADS * C0_IPT));
    if (blocks == 0) return;
    seg_compact0_kernel<<<blocks, C0_THREADS, 0, st>>>(flags, sidx, m, carry_head, carry_keep, cpos, cidx, cgrp);
}

// ---------------------------------------------------------------- group-local refinement (no radix sort)
// After round 0 nearly all surviving groups hold two or three suffixes.  Sorting them with seven or eight radix
// passes over the whole working set is out of proportion: here every small group is ordered by comparing the text
// directly from the known depth on (up to GS_DEPTH more symbols; the end of the text is smallest), written back in
// order, and every element gets the key (group start << 32 | number of its sub-group): equal keys = still tied within
// GS_DEPTH symbols.  The usual
// seg_reduce / seg_scan / seg_apply then refine on these keys.  Groups above GS_MAX elements are left alone (one key
// for the whole group): they go to the next regular round, whose depth therefore stays where it was.
// -1 / 0 / +1: order of suffixes a and b beyond the `depth` symbols they share, 0 = tied within GS_DEPTH symbols
__device__ __forceinline__ int suffix_cmp_from(const uint8_t *__restrict__ text, uint64_t n, uint64_t a, uint64_t b,
                                               uint64_t depth)
{
    uint64_t pa = a + depth, pb = b + depth;
    for (int q = 0; q < GS_DEPTH; ++q, ++pa, ++pb) {
        if (pa >= n || pb >= n) {
            if (pa >= n && pb >= n) return a > b ? -1 : 1;      // both ended: the shorter suffix (larger id) is smaller
            return pa >= n ? -1 : 1;
        }
        const uint32_t ca = text[pa], cb = text[pb];
        if (ca != cb) return ca < cb ? -1 : 1;
    }
    return 0;
}

// One group of s <= GS_MAX elements starting at element j, ordered by ONE thread with symbol-by-symbol comparisons
// (GS_DEPTH deep, end of text exact).  The general case; group_sort_kernel sends here only what its 24-byte windows
// cannot decide.
template <bool WIDE>
__device__ __forceinline__ void group_sort_serial(uint32_t *__restrict__ cidx, uint32_t j, uint32_t s, uint32_t g,
                                               const uint8_t *__restrict__ text, uint64_t n, uint64_t depth,
                                               const uint64_t *__restrict__ ids64, uint64_t *__restrict__ keys)
{
    uint32_t v[GS_MAX];                                         // cidx entries (suffix ids, or ordinals when WIDE)
    uint64_t id[GS_MAX];
    for (uint32_t i = 0; i < s; ++i) {
        v[i] = cidx[j + i];
        id[i] = WIDE ? (ids64[v[i]] & WIDE_ID_MASK) : (uint64_t)v[i];
    }
    for (uint32_t i = 1; i < s; ++i) {                          // insertion sort: groups are tiny
        const uint32_t xv = v[i];
        const uint64_t xi = id[i];
        uint32_t k = i;
        while (k > 0 && suffix_cmp_from(text, n, xi, id[k - 1], depth) < 0) {
            v[k] = v[k - 1];
            id[k] = id[k - 1];
            --k;
        }
        v[k] = xv;
        id[k] = xi;
    }
    uint32_t sub = 0;
    for (uint32_t i = 0; i < s; ++i) {
        if (i > 0 && suffix_cmp_from(text, n, id[i - 1], id[i], depth) != 0) ++sub;
        cidx[j + i] = v[i];
        keys[j + i] = ((uint64_t)g << 32) | sub;
    }
}

// the 8 * WW symbols at text[p .. p + 8 WW) as WW big-endian words (integer order = symbol order); WW + 1 aligned
// 8-byte loads, all inside [p - 7, p + 8 WW + 8)
__device__ __forceinline__ uint64_t be64(uint64_t x)
{
    return ((uint64_t)__byte_perm((uint32_t)x, 0u, 0x0123) << 32) | __byte_perm((uint32_t)(x >> 32), 0u, 0x0123);
}
template <int WW>
__device__ __forceinline__ void window_be(const uint8_t *__restrict__ text, uint64_t p, uint64_t w[WW])
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(text) + p;
    const uint64_t *g = reinterpret_cast<const uint64_t *>(a & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(a & 7u) * 8u;
    uint64_t x[WW + 1];
#pragma unroll
    for (int q = 0; q <= WW; ++q) x[q] = __ldg(g + q);
#pragma unroll
    for (int q = 0; q < WW; ++q) w[q] = be64(sh ? (x[q] >> sh) | (x[q + 1] << (64u - sh)) : x[q]);
}

// One thread per ELEMENT (the one-thread-per-group form left two thirds of the lanes idle behind serial chains of
// dependent random loads and kept its arrays in local memory: 164 M elements took 8 ms, the distributed build's group
// round 13-44 ms).  A CTA takes 1008 elements + 16 of look-ahead: (1) group ids into shared memory, every element
// finds its group's start and size by scanning at most 16 neighbours; a group of 2..16 elements belongs to the CTA
// holding its first element, larger groups keep one key (g << 32); (2) every member loads its suffix id and the 8 WW
// symbols beyond the shared depth as WW big-endian words -- two dependent random loads per element, all elements in
// flight at once; (3) place in the group = members with a smaller window, key = (g << 32 | that count).  Groups with
// two equal windows (ties deeper than 8 WW symbols) or a window reaching the end of the text go to
// group_sort_serial on the thread of their first element: the result is that of the serial form in every case.
// WW = 2 (16 symbols) where the uniform depth is about what equal keys share (per-symbol keys: C3's 9 of ~10); WW = 3
// for k-gram keys, which guarantee one gram but share ~3 (C2: 6 symbols guaranteed, 18-21 shared): with 16 symbols
// nearly every group tied and went to the serial form (C2 group round 0.078 ms, 0.060 with 24; on C3, 24 symbols cost
// more loads than they save: 14.33 -> 14.42 ms per build; B200, 1000 W).
constexpr int GC_THREADS = 256;
constexpr int GC_IPT = 4;
constexpr int GC_SLOTS = GC_THREADS * GC_IPT;        // 1024 elements seen by a CTA
constexpr int GC_HALO = GS_MAX;                      // look-ahead (and look-back for the group ids)
constexpr int GC_STRIDE = GC_SLOTS - GC_HALO;        // elements owned by a CTA
constexpr uint32_t GC_NOGROUP = 0xFFFFFFFFu;         // group ids are positions < 2^30
constexpr uint32_t GC_MARK = 0xFFFFFFFFu;            // low key word of a group's first element: "order me serially"
constexpr int GC_WORDS = (GC_SLOTS + 2 * GC_HALO) / 32;
static_assert((GC_SLOTS + 2 * GC_HALO) % 32 == 0 && GC_HALO <= 32, "start bits are read one word back and one ahead");

template <bool WIDE, int WW>
__global__ void __launch_bounds__(GC_THREADS, 6)
group_sort_kernel(uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp, uint32_t m,
                  const uint8_t *__restrict__ text, uint64_t n, uint64_t depth, const uint64_t *__restrict__ ids64,
                  uint64_t *__restrict__ keys)
{
    __shared__ uint32_t s_grp[GC_SLOTS + 2 * GC_HALO];           // element base - GC_HALO + i
    __shared__ uint64_t s_w[WW][GC_SLOTS];                       // the window, most significant word first
    __shared__ uint32_t s_v[GC_SLOTS];
    __shared__ uint16_t s_meta[GC_SLOTS];                        // start slot (10 bits) | size - 1 (4 bits) | member (bit 15)
    __shared__ uint16_t s_x[WIDE ? GC_SLOTS : 1];                // WIDE: the key's extension bits out of the id word
    __shared__ uint8_t s_hard[GC_SLOTS];                         // this member's window cannot decide its place
    __shared__ uint32_t s_headw[GC_WORDS + 2];                   // group-start bits of the positions in s_grp
    const uint32_t tid = threadIdx.x;
    const uint32_t base = blockIdx.x * (uint32_t)GC_STRIDE;
    for (uint32_t i = tid; i < GC_SLOTS + 2 * GC_HALO; i += GC_THREADS) {
        const int64_t e = (int64_t)base - GC_HALO + i;
        s_grp[i] = (e >= 0 && e < (int64_t)m) ? cgrp[e] : GC_NOGROUP;
    }
    __syncthreads();
    // one bit per position: "a group starts here" (position 0 counts as a start: whatever begins before the look-back
    // is 16 or more away from every element this CTA decides on)
    for (uint32_t i = tid; i < GC_SLOTS + 2 * GC_HALO; i += GC_THREADS) {
        const uint32_t word = __ballot_sync(0xffffffffu, i == 0 || s_grp[i] != s_grp[i - 1]);
        if ((tid & 31u) == 0) s_headw[i >> 5] = word;
    }
    if (tid == 0) s_headw[GC_WORDS] = s_headw[GC_WORDS + 1] = 0xFFFFFFFFu;     // past the end: every position a start
    __syncthreads();
#pragma unroll 2
    for (int k = 0; k < GC_IPT; ++k) {
        const uint32_t slot = k * GC_THREADS + tid;
        const uint32_t e = base + slot;
        uint16_t meta = 0;
        if (e < m) {
            const uint32_t g = s_grp[GC_HALO + slot];
            // start of the group = the last start bit at or before this position, its end = the next one after it:
            // two words of bits decide both (a group of up to 16 spans at most two words); farther = "more than 16"
            const uint32_t pos = GC_HALO + slot, w = pos >> 5, b = pos & 31u;
            const uint32_t le = 0xFFFFFFFFu >> (31u - b);                         // bits 0..b
            const uint32_t cur = s_headw[w];
            uint32_t st;
            if (cur & le) st = (w << 5) + 31u - __clz(cur & le);
            else { const uint32_t prev = s_headw[w - 1]; st = prev ? ((w - 1) << 5) + 31u - __clz(prev) : 0u; }
            uint32_t nx;
            if (cur & ~le) nx = (w << 5) + __ffs(cur & ~le) - 1u;
            else { const uint32_t nxt = s_headw[w + 1]; nx = nxt ? ((w + 1) << 5) + __ffs(nxt) - 1u : pos + GS_MAX + 1u; }
            const uint32_t size = min(nx - st, (uint32_t)GS_MAX + 1u);           // GS_MAX + 1 = "more than GS_MAX"
            const int start = (int)st - GC_HALO;
            if (size < 2 || size > (uint32_t)GS_MAX) {
                if (slot < (uint32_t)GC_STRIDE) keys[e] = (uint64_t)g << 32;      // left to the next regular round
            } else if (start >= 0 && start < GC_STRIDE) {
                const uint32_t v = cidx[e];
                uint64_t id = v;
                if (WIDE) {
                    const uint64_t w = ids64[v];
                    id = w & WIDE_ID_MASK;
                    s_x[slot] = (uint16_t)(w >> WIDE_ID_BITS);
                }
                s_w[0][slot] = id + depth;                       // where this member's window starts (until the window itself lands here)
                s_v[slot] = v;
                meta = (uint16_t)(0x8000u | ((size - 1) << 10) | (uint32_t)start);
            }
        }
        s_meta[slot] = meta;
    }
    __syncthreads();
    // the window: 8 WW symbols beyond the shared depth -- for 64-bit ids only where the extension bits of the key
    // (16 more bits of the code stream, carried in the id word) do not already tell this member from all the others
#pragma unroll 2
    for (int k = 0; k < GC_IPT; ++k) {
        const uint32_t slot = k * GC_THREADS + tid;
        const uint32_t meta = s_meta[slot];
        uint8_t hard = 0;
        if (meta & 0x8000u) {
            bool need = true;
            if (WIDE) {
                const uint32_t start = meta & 0x3FFu, size = ((meta >> 10) & 0xFu) + 1;
                const uint16_t x = s_x[slot];
                need = false;
                for (uint32_t i = 0; i < size; ++i) need |= (start + i != slot && s_x[start + i] == x);
            }
            uint64_t w[WW];
#pragma unroll
            for (int q = 0; q < WW; ++q) w[q] = 0;
            if (need) {
                const uint64_t p = s_w[0][slot];
                if (p >= 8 && p + 8 * (WW + 1) <= n) window_be<WW>(text, p, w);
                else hard = 1;
            }
#pragma unroll
            for (int q = 0; q < WW; ++q) s_w[q][slot] = w[q];
        }
        s_hard[slot] = hard;
    }
    __syncthreads();
    // place among the members; a member whose window equals another member's marks the group as hard
    uint32_t place[GC_IPT], less[GC_IPT];
#pragma unroll
    for (int k = 0; k < GC_IPT; ++k) {
        const uint32_t slot = k * GC_THREADS + tid;
        const uint32_t meta = s_meta[slot];
        place[k] = less[k] = 0;
        if (!(meta & 0x8000u)) continue;
        const uint32_t start = meta & 0x3FFu, size = ((meta >> 10) & 0xFu) + 1;
        uint64_t w[WW];
#pragma unroll
        for (int q = 0; q < WW; ++q) w[q] = s_w[q][slot];
        const uint32_t x = WIDE ? s_x[slot] : 0u;
        bool tie = false;
        for (uint32_t i = 0; i < size; ++i) {
            const uint32_t o = start + i;
            if (o == slot) continue;
            const uint32_t ox = WIDE ? s_x[o] : 0u;
            // lexicographic over (extension bits, window words): the first word that differs decides
            bool eq = ox == x, lt = ox < x;
#pragma unroll
            for (int q = 0; q < WW; ++q) {
                const uint64_t ow = s_w[q][o];
                lt |= eq && ow < w[q];
                eq &= ow == w[q];
            }
            tie |= eq;
            less[k] += lt;
            place[k] += lt || (eq && o < slot);
        }
        if (tie) s_hard[slot] = 1;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GC_IPT; ++k) {
        const uint32_t slot = k * GC_THREADS + tid;
        const uint32_t meta = s_meta[slot];
        if (!(meta & 0x8000u)) continue;
        const uint32_t start = meta & 0x3FFu, size = ((meta >> 10) & 0xFu) + 1;
        bool hard = false;
        for (uint32_t i = 0; i < size; ++i) hard |= (s_hard[start + i] != 0);
        const uint32_t g = s_grp[GC_HALO + slot];
        if (hard) {       // left to group_sort_marked_kernel: the first element's key carries the mark
            keys[base + slot] = ((uint64_t)g << 32) | (slot == start ? GC_MARK : 0u);
            continue;
        }
        const uint32_t out = base + start + place[k];
        cidx[out] = s_v[slot];
        keys[out] = ((uint64_t)g << 32) | less[k];
    }
}

// second launch of the element-parallel form: the groups it marked (windows that tie or reach the end of the text)
// ordered serially by the thread of their first element; everybody else reads one key and leaves
template <bool WIDE>
__global__ void __launch_bounds__(256)
group_sort_marked_kernel(uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp, uint32_t m,
                         const uint8_t *__restrict__ text, uint64_t n, uint64_t depth,
                         const uint64_t *__restrict__ ids64, uint64_t *__restrict__ keys)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint64_t k = keys[j];
    if ((uint32_t)k != GC_MARK) return;
    const uint32_t g = (uint32_t)(k >> 32);
    uint32_t s = 1;
    while (s < (uint32_t)GS_MAX && j + s < m && cgrp[j + s] == g) ++s;
    group_sort_serial<WIDE>(cidx, j, s, g, text, n, depth, ids64, keys);
}

cudaError_t group_local_keys(uint32_t *cidx, const uint32_t *cgrp, uint32_t m, const uint8_t *text, uint64_t n,
                             uint64_t depth, bool gram_keys, const uint64_t *ids64, uint64_t *keys, cudaStream_t st)
{
    if (m == 0) return cudaSuccess;
    const uint32_t blocks = (m + GC_STRIDE - 1) / GC_STRIDE;
    const uint32_t blocks2 = (m + 255) / 256;
    if (ids64) {
        group_sort_kernel<true, 2><<<blocks, GC_THREADS, 0, st>>>(cidx, cgrp, m, text, n, depth, ids64, keys);
        group_sort_marked_kernel<true><<<blocks2, 256, 0, st>>>(cidx, cgrp, m, text, n, depth, ids64, keys);
    } else {
        if (gram_keys) group_sort_kernel<false, 3><<<blocks, GC_THREADS, 0, st>>>(cidx, cgrp, m, text, n, depth, ids64, keys);
        else group_sort_kernel<false, 2><<<blocks, GC_THREADS, 0, st>>>(cidx, cgrp, m, text, n, depth, ids64, keys);
        group_sort_marked_kernel<false><<<blocks2, 256, 0, st>>>(cidx, cgrp, m, text, n, depth, ids64, keys);
    }
    count_launch(2);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- the last, tiny rounds in one CTA
// Once at most FIN_MAX suffixes are left (C2: 6 after two rounds, C3: 20) a round of the general path is ~25 launches
// and two host round trips for nothing.  One CTA finishes the job on its own: key build (same look-ups), bitonic sort
// of the (group, rank) keys in shared memory, head flags, SA / rank writes, compaction, doubling -- until every group
// is a singleton.  Same recurrences as sa_keybuild_kernel + the radix sort + seg_* kernels.
constexpr int FIN_MAX = 1024;

__global__ void __launch_bounds__(FIN_MAX)
sa_finish_small_kernel(const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp,
                       const uint32_t *__restrict__ cpos, uint32_t m, uint32_t n, uint64_t h, uint32_t *sa,
                       uint32_t *rank, LazyRank lz, AlphaCode ac, const uint8_t *__restrict__ text,
                       uint8_t *__restrict__ bwt)
{
    __shared__ uint64_t s_key[FIN_MAX];
    __shared__ uint32_t s_idx[FIN_MAX], s_grp[FIN_MAX], s_pos[FIN_MAX], s_aux[FIN_MAX];
    __shared__ AlphaKeys::Tab s_tab;
    __shared__ uint32_t s_w[32], s_w2[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    s_tab.load(ac);
    if (tid < m) { s_idx[tid] = cidx[tid]; s_grp[tid] = cgrp[tid]; s_pos[tid] = cpos[tid]; }
    __syncthreads();
    for (int iter = 0; iter < 64 && m > 0; ++iter) {
        // ---- keys: (group start, rank of the suffix h symbols later + 1), padding sorts last
        uint64_t key = ~0ULL;
        uint32_t idx = 0;
        if (tid < m) {
            idx = s_idx[tid];
            const uint64_t t = (uint64_t)idx + h;
            uint32_t k2 = 0;
            if (t < n)
                k2 = (lz.text ? lazy_rank_lookup<true>(lz, s_tab, n, (uint32_t)t, rank)
                              : *reinterpret_cast<const volatile uint32_t *>(rank + t)) + 1u;
            key = ((uint64_t)s_grp[tid] << 32) | k2;
        }
        s_key[tid] = key;
        s_aux[tid] = idx;
        __syncthreads();
        // ---- bitonic sort of (key, suffix id): equal keys stay one group, their order inside does not matter
        for (uint32_t k = 2; k <= FIN_MAX; k <<= 1) {
            for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                const uint32_t partner = tid ^ j;
                if (partner > tid) {
                    const uint64_t a = s_key[tid], b = s_key[partner];
                    const bool up = (tid & k) == 0;
                    if ((a > b) == up) {
                        s_key[tid] = b; s_key[partner] = a;
                        const uint32_t x = s_aux[tid]; s_aux[tid] = s_aux[partner]; s_aux[partner] = x;
                    }
                }
                __syncthreads();
            }
        }
        key = s_key[tid];
        idx = s_aux[tid];
        const bool in = tid < m;
        const bool head = in && (tid == 0 || key != s_key[tid - 1]);
        const bool next_head = (tid + 1 >= m) || (s_key[tid + 1] != key);
        const bool single = head && next_head;
        // ---- group start = slot of the governing head (inclusive max-scan of head indices over the block)
        uint32_t hv = head ? tid + 1 : 0u;
        hv = warp_incl_max(hv);
        if (lane == 31) s_w[warp] = hv;
        // ---- compaction slots of the non-singletons (exclusive sum-scan)
        const uint32_t keep = (in && !single) ? 1u : 0u;
        uint32_t wtot;
        const uint32_t ex = warp_excl_sum(keep, wtot);
        if (lane == 31) s_w2[warp] = wtot;
        __syncthreads();
        uint32_t ph = 0, pk = 0, total = 0;
        for (uint32_t w = 0; w < FIN_MAX / 32; ++w) {
            if (w < warp) { ph = max(ph, s_w[w]); pk += s_w2[w]; }
            total += s_w2[w];
        }
        const uint32_t gslot = max(ph, hv);                     // (index of the governing head) + 1
        const uint32_t p = in ? s_pos[tid] : 0u;
        const uint32_t newgrp = in ? s_pos[gslot - 1] : 0u;
        __syncthreads();                                        // every thread has read s_pos / s_key
        if (in) {
            sa[p] = idx;
            if (bwt) bwt[p] = text[idx ? idx - 1u : n - 1u];
            *reinterpret_cast<volatile uint32_t *>(rank + idx) = newgrp;
        }
        if (keep) {
            const uint32_t slot = pk + ex;
            s_idx[slot] = idx;
            s_grp[slot] = newgrp;
            s_aux[slot] = p;                                    // the new slot list, moved to s_pos below
        }
        __threadfence_block();
        __syncthreads();
        if (tid < total) s_pos[tid] = s_aux[tid];
        m = total;
        h *= 2;
        lz.first_round = 0;
        __syncthreads();
    }
}

}  // namespace hkcsa

// ------------------------------------------------------------------ host driver
using namespace hkcsa;

namespace {
struct SaBuffers {
    uint64_t *key[2];
    uint32_t *val[2];
    uint32_t *pos[2];
    uint32_t *grp;
    uint32_t *rank;
    uint32_t *agg_head, *agg_keep;
    uint16_t *flags;
    uint32_t *counter;
    uint64_t *hist64;
    uint32_t *bucket;
    uint64_t *samples;
    GramScratch gram;
    SortScratch sort;
};

SaBuffers carve_sa(Carver &c, uint64_t n)
{
    SaBuffers b;
    const uint64_t tiles = (n + SEG_TILE - 1) / SEG_TILE + 1;
    b.key[0] = c.take<uint64_t>(n);
    b.key[1] = c.take<uint64_t>(n);
    b.val[0] = c.take<uint32_t>(n);
    b.val[1] = c.take<uint32_t>(n);
    b.pos[0] = c.take<uint32_t>(n);
    b.pos[1] = c.take<uint32_t>(n);
    b.grp = c.take<uint32_t>(n);
    b.rank = c.take<uint32_t>(n);
    b.agg_head = c.take<uint32_t>(tiles);
    b.agg_keep = c.take<uint32_t>(tiles);
    b.flags = c.take<uint16_t>(tiles * SEG_THREADS);
    b.counter = c.take<uint32_t>(64);
    b.hist64 = c.take<uint64_t>(256);
    b.bucket = c.take<uint32_t>((1u << LAZY_BUCKET_BITS) + 2);
    b.samples = c.take<uint64_t>((n >> LAZY_SAMPLE_SHIFT) + 2);
    b.gram.tab = c.take<uint32_t>(GRAM_MAX_G);
    b.gram.hist = c.take<uint32_t>(GRAM_MAX_G);
    b.gram.cum = c.take<uint64_t>(GRAM_MAX_G + 8 + GRAM_MAX_CHUNKS + 8);      // per-chunk prefix sums, then the chunk totals
    b.gram.stats = c.take<uint64_t>(8);
    b.sort = carve_sort_scratch(c, n);
    return b;
}
}  // namespace

extern "C" size_t hkcsa_sa_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    carve_sa(c, n);
    return c.total();
}

extern "C" int hkcsa_byte_hist(const uint8_t *d_sym, uint64_t n, uint64_t *d_hist, void *stream)
{
    HK_REQUIRE(d_hist != nullptr && (d_sym != nullptr || n == 0), HKCSA_EINVAL, "null pointer");
    HK_CUDA(byte_hist(d_sym, n, d_hist, as_stream(stream)));
    return HKCSA_OK;
}

// d_bwt != nullptr: the BWT (csa/bwt.py:3-13) is produced along with the suffix array.  With round-0 keys of at most
// 56 bits the symbol before each suffix rides through the sort in the top byte of its key, seg_reduce_kernel writes the
// rows as it reads the sorted keys, and the rounds that move a suffix to its final slot rewrite that slot's row; with
// 64-bit keys the phased gather of bwt.cu runs after the build.
static int sa_build_impl(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint8_t *d_bwt, void *d_scratch,
                         size_t scratch_bytes, void *stream, hkcsa_sa_stats *h_stats)
{
    hkcsa_sa_stats stats;
    memset(&stats, 0, sizeof(stats));
    if (h_stats) *h_stats = stats;
    if (n == 0) return HKCSA_OK;   // build_suffix_array("") == []
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    HK_REQUIRE(d_text && d_sa && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(((reinterpret_cast<uintptr_t>(d_sa) | reinterpret_cast<uintptr_t>(d_scratch)) & 15) == 0, HKCSA_EINVAL,
               "d_sa and d_scratch must be 16-byte aligned (TMA bulk copies)");
    Carver c(d_scratch);
    SaBuffers B = carve_sa(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "SA scratch too small");
    cudaStream_t st = as_stream(stream);
    uint8_t *pin = static_cast<uint8_t *>(pinned_page());
    HK_REQUIRE(pin != nullptr, HKCSA_ECUDA, "pinned page allocation failed");
    uint64_t *h_hist = reinterpret_cast<uint64_t *>(pin);           // 2048 bytes
    uint32_t *h_m = reinterpret_cast<uint32_t *>(pin + 2048);

    // ---- alphabet: dense codes 1..sigma in byte order, 0 = past the end
    HK_CUDA(byte_hist(d_text, n, B.hist64, st));
    HK_CUDA(cudaMemcpyAsync(h_hist, B.hist64, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    static thread_local Round0Plan r0;
    if (int rc = plan_round0(h_hist, r0, d_text, n, &B.gram, st)) return rc;
    const AlphaCode &ac = r0.ac;
    const GramCode &gc = r0.gram;
    const uint32_t sigma = r0.sigma;
    const uint32_t N = (uint32_t)n;
    stats.gram_k = gc.tab ? gc.k : 0;
    const int max_len = r0.max_len, bits0 = r0.bits0, k0 = r0.k0, passes0 = r0.passes0;
    stats.sigma = sigma;
    memcpy(stats.byte_hist, h_hist, sizeof(stats.byte_hist));
    stats.bits_per_symbol = (uint32_t)max_len;
    stats.k0 = (uint32_t)k0;
    stats.key_bits0 = (uint32_t)bits0;
    const bool carry = d_bwt != nullptr && bits0 <= 56;
    stats.bwt_carried = carry ? 1u : 0u;
    const uint64_t mask0 = bits0 >= 64 ? ~0ULL : ((1ULL << bits0) - 1ULL);

    HK_CUDA(cudaMemsetAsync(B.sort.hist, 0, 8 * RADIX * sizeof(uint32_t), st));
    // Round 0.  The value ping-pong is (d_sa, val[0]) arranged so the sorted suffix ids land in d_sa:
    // the suffix array of round 0 needs no extra copy.
    uint64_t *ka = B.key[0], *kb = B.key[1];
    uint32_t *va = (passes0 % 2 == 0) ? d_sa : B.val[0];
    uint32_t *vb = (passes0 % 2 == 0) ? B.val[0] : d_sa;
    {
        prof::Scope ps(st, prof::SA_PACK0, (uint64_t)N * 9);
        if (gc.tab) launch_pack0(GramKeys{gc}, passes0, carry, d_text, N, ka, B.sort.hist, st);
        else launch_pack0(AlphaKeys{ac, (uint32_t)max_len}, passes0, carry, d_text, N, ka, B.sort.hist, st);
        HK_LAUNCH_CHECK();
    }
    HK_CUDA(radix_sort_pairs_u64(ka, va, kb, vb, N, passes0, B.sort, st, /*identity_vals=*/true));
    uint64_t *skey = (passes0 % 2 == 0) ? ka : kb;     // sorted round-0 keys
    uint64_t *kfree = (passes0 % 2 == 0) ? kb : ka;
    uint32_t *sidx = d_sa;                              // sorted suffix ids
    uint32_t m = N;
    const uint32_t *pos = nullptr;                      // SA slots of the working set (round 0: identity)
    int pcur = 0;
    uint64_t h = (uint64_t)k0;
    const int b2 = (int)bits_for(n);           // rank + 1 <= n
    const int b1 = (int)bits_for(n - 1);       // group start <= n - 1
    uint32_t round = 0;
    stats.round_elems[0] = m;
    stats.round_passes[0] = (uint32_t)passes0;
    stats.sort_elem_passes = (uint64_t)m * passes0;
    stats.alg_bytes = (uint64_t)n * 9 + (uint64_t)m * (24ull * passes0) - (uint64_t)m * 4;   // pass 0 reads no ids

    LazyRank lz;
    lz.text = nullptr; lz.keys0 = nullptr; lz.bucket = nullptr; lz.samples = nullptr; lz.first_round = 0; lz.bits = bits0;
    const int bucket_bits = std::min(LAZY_BUCKET_BITS, bits0);
    lz.shift = bits0 - bucket_bits;
    lz.mask = mask0;
    lz.gram = GramKeys{gc};
    uint64_t *kx = nullptr, *ky = nullptr;             // key ping-pong of the later rounds
    uint32_t *vfree = B.val[1];                        // free value buffer (receives the compacted ids)
    uint32_t *vother = B.val[0];                       // the round-0 sort's other value buffer: free from here on

    bool lazy_index_due = false;
    // the look-up structures over the sorted round-0 keys (lz.keys0): built on first use -- when the group-local
    // round finishes the job no look-up ever happens
    auto build_lazy_index = [&]() -> int {
        if (!lazy_index_due) return HKCSA_OK;
        lazy_index_due = false;
        const uint32_t nbuckets = 1u << bucket_bits;
        prof::Scope ps(st, prof::OTHER, (uint64_t)nbuckets * 8);
        sa_bucket_index_kernel<<<(nbuckets + 1 + 255) / 256, 256, 0, st>>>(lz.keys0, N, lz.shift, lz.mask, nbuckets,
                                                                           B.bucket);
        HK_LAUNCH_CHECK();
        const uint32_t nsamp = (uint32_t)(((uint64_t)N + (1u << LAZY_SAMPLE_SHIFT) - 1) >> LAZY_SAMPLE_SHIFT);
        sa_key_samples_kernel<<<(nsamp + 255) / 256, 256, 0, st>>>(lz.keys0, N, lz.mask, B.samples);
        HK_LAUNCH_CHECK();
        return HKCSA_OK;
    };
    while (true) {
        // ---- refine ranks from the sorted keys
        const uint32_t tiles = (m + SEG_TILE - 1) / SEG_TILE;
        {
            const bool emit = carry && round == 0;      // round 0: the sorted keys deliver the BWT
            prof::Scope ps(st, prof::SEG_REDUCE, (uint64_t)m * 8 + m / 4 + (emit ? m : 0));
            seg_reduce_kernel<<<tiles, SEG_THREADS, 0, st>>>(skey, m, B.agg_head, B.agg_keep, B.flags,
                                                             round == 0 ? mask0 : ~0ULL, emit ? d_bwt : nullptr);
            HK_LAUNCH_CHECK();
        }
        {
            prof::Scope ps(st, prof::SEG_SCAN, (uint64_t)tiles * 16);
            seg_scan_kernel<<<1, 1024, 0, st>>>(B.agg_head, B.agg_keep, tiles, B.counter);
            HK_LAUNCH_CHECK();
        }
        HK_CUDA(cudaMemcpyAsync(h_m, B.counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        HK_CUDA(cudaStreamSynchronize(st));
        const uint32_t m_next = *h_m;
        bool scatter_all = true;
        if (round == 0 && m_next > 0 && (uint64_t)m_next * 4 <= n) {
            // few survivors: scatter ranks only for them, look the others up on demand
            lz.text = d_text;
            lz.keys0 = skey;
            lz.bucket = B.bucket;
            scatter_all = false;
            lz.samples = B.samples;
            lazy_index_due = true;          // bucket index + key samples are built when a look-up round actually comes
            stats.lazy_ranks = 1;
        }
        uint32_t *cpos = B.pos[pcur ^ 1];
        uint32_t *cidx = vfree;
        {
            // flags + (round 0, lazy ranks: survivors only; otherwise ids, slots, rank scatter)
            prof::Scope ps(st, prof::SEG_APPLY, m / 4 + (uint64_t)m_next * 20 +
                                                 ((round != 0 || scatter_all) ? (uint64_t)m * 12 : 0));
            // round 0 with lazy ranks writes no ranks at all: round 1 takes them from the look-up (group start =
            // lower bound), and round 1's own scatter covers every survivor before round 2 reads the array.  After
            // the last round nothing reads the ranks.
            if (round == 0 && !scatter_all) {
                seg_compact0(B.flags, sidx, m, B.agg_head, B.agg_keep, cpos, cidx, B.grp, st);
            } else {
                seg_apply_kernel<<<tiles, SEG_THREADS, 0, st>>>(B.flags, sidx, pos, m, B.agg_head, B.agg_keep, d_sa,
                                                               m_next == 0 ? nullptr : B.rank, cpos, cidx, B.grp,
                                                               round != 0, scatter_all, d_text, N,
                                                               carry ? d_bwt : nullptr);
            }
            HK_LAUNCH_CHECK();
        }
        stats.alg_bytes += (uint64_t)m * 8 + m / 2 + (uint64_t)m_next * 20 + ((round != 0 || scatter_all) ? (uint64_t)m * 12 : 0);
        ++round;
        if (m_next == 0) break;
        HK_REQUIRE(h < n, HKCSA_EINVAL, "internal: groups remain after depth >= n");
        HK_REQUIRE(round < 40, HKCSA_EINVAL, "internal: too many doubling rounds");
        if (m_next <= (uint32_t)FIN_MAX) {
            // the few suffixes left are finished by one CTA: no more launches per round, no more host round trips
            lz.first_round = (round == 1) ? 1 : 0;
            if (int rc = build_lazy_index()) return rc;
            prof::Scope ps(st, prof::OTHER, (uint64_t)m_next * 32);
            sa_finish_small_kernel<<<1, FIN_MAX, 0, st>>>(cidx, B.grp, cpos, m_next, N, std::min<uint64_t>(h, n), d_sa,
                                                          B.rank, lz, ac, d_text, carry ? d_bwt : nullptr);
            HK_LAUNCH_CHECK();
            stats.round_elems[round] = m_next;
            stats.round_passes[round] = 0;                      // 0 passes = finished in shared memory
            ++round;
            break;
        }
        // ---- buffers of the next round
        if (round == 1) {
            if (lz.text) { kx = kfree; ky = kfree + align_up(m_next, 32); }   // round-0 keys stay intact; 16-byte aligned for TMA
            else { kx = kfree; ky = skey; }
            vother = B.val[0];
        } else {
            vother = sidx;                                     // the sorted ids just consumed: free again
        }
        m = m_next;
        pcur ^= 1;
        pos = B.pos[pcur];
        uint32_t *vx = cidx, *vy = vother;
        if (round == 1 && (uint64_t)m * 2 <= n && !getenv("HKCSA_NO_GROUP_ROUND")) {
            // Round 1 without a radix sort: the survivors of round 0 sit in groups of two or three; each small group
            // is ordered by comparing text beyond the k0 symbols its members share.  The depth does not advance
            // (large groups are untouched), every survivor gets its rank scattered by the refinement that follows.
            prof::Scope ps(st, prof::SA_KEYBUILD, (uint64_t)m * 48);
            HK_CUDA(group_local_keys(vx, B.grp, m, d_text, n, std::min<uint64_t>(h, n), gc.tab != nullptr, nullptr, kx, st));
            skey = kx; sidx = vx; vfree = vy;
            stats.round_elems[round] = m;
            stats.round_passes[round] = 0;                      // 0 passes = refined without a radix sort
            stats.alg_bytes += (uint64_t)m * 48;
            continue;
        }
        const int bits = b1 + b2;
        const int passes = (bits + 7) / 8;
        HK_CUDA(cudaMemsetAsync(B.sort.hist, 0, 8 * RADIX * sizeof(uint32_t), st));
        lz.first_round = (round == 1) ? 1 : 0;
        if (int rc = build_lazy_index()) return rc;
        {
            const int blocks = (int)std::min<uint64_t>(((uint64_t)m + 255) / 256, (uint64_t)num_sms() * 16);
            prof::Scope ps(st, prof::SA_KEYBUILD, (uint64_t)m * 20);
            sa_keybuild_kernel<<<blocks, 256, 0, st>>>(vx, B.grp, B.rank, N, (uint32_t)std::min<uint64_t>(h, n), b2,
                                                       m, passes, kx, B.sort.hist, lz, ac);
            HK_LAUNCH_CHECK();
        }
        HK_CUDA(radix_sort_pairs_u64(kx, vx, ky, vy, m, passes, B.sort, st));
        if (passes & 1) { skey = ky; sidx = vy; vfree = vx; }
        else { skey = kx; sidx = vx; vfree = vy; }
        stats.round_elems[round] = m;
        stats.round_passes[round] = (uint32_t)passes;
        stats.sort_elem_passes += (uint64_t)m * passes;
        stats.alg_bytes += (uint64_t)m * (20ull + 24ull * passes);
        h *= 2;
    }
    stats.rounds = round;
    if (carry) stats.alg_bytes += n;
    if (h_stats) *h_stats = stats;
    if (d_bwt && !carry) return bwt_gather(d_text, d_sa, n, d_bwt, st);
    return HKCSA_OK;
}

extern "C" int hkcsa_sa_build(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, void *d_scratch,
                              size_t scratch_bytes, void *stream, hkcsa_sa_stats *h_stats)
{
    return sa_build_impl(d_text, n, d_sa, nullptr, d_scratch, scratch_bytes, stream, h_stats);
}

extern "C" int hkcsa_sa_bwt_build(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint8_t *d_bwt, void *d_scratch,
                                  size_t scratch_bytes, void *stream, hkcsa_sa_stats *h_stats)
{
    HK_REQUIRE(d_bwt != nullptr || n == 0, HKCSA_EINVAL, "null pointer");
    return sa_build_impl(d_text, n, d_sa, d_bwt, d_scratch, scratch_bytes, stream, h_stats);
}
