// suffix_array.cuh -- pieces of K1 shared by the single-GPU builder (suffix_array.cu) and the distributed
// builder (dist_sa.cu): the order-preserving prefix codes of round 0, the round-0 plan, the key sources that make the
// round-0 keys, and the segmented rank-update kernels.
#pragma once
#include "common.cuh"
#include "radix_sort.cuh"

namespace hkcsa {

constexpr int SEG_THREADS = 256;
constexpr int SEG_IPT = 8;
constexpr int SEG_TILE = SEG_THREADS * SEG_IPT;

struct CodeMap {
    uint16_t code[256];  // byte -> dense code + 1 (0 for bytes that do not occur)
};

// Order-preserving prefix code ("alphabetic code") over {past-the-end} + the symbols of the text: frequent
// symbols get short codes, and comparing two code streams bit by bit equals comparing the symbol strings,
// the end of the text being smallest.  The round-0 key of a suffix is the first `bits` bits of its code
// stream, so a key covers as many symbols as a fixed-width packing would in fewer bits -- fewer radix passes
// (DNA + '$': 21 symbols in 48 bits instead of 63).  Equal keys share at least bits / max_len symbols.
struct AlphaCode {
    uint32_t code[257];   // right-aligned; [256] = past the end
    uint8_t len[257];
};

// returns false when the code would be degenerate (then the caller keeps fixed-width codes)
bool build_alpha_code(const uint64_t *h_hist, AlphaCode &ac, double &avg_len, int &max_len);

// The same idea over k-GRAMS (single-GPU builder): the order-preserving prefix code is built over the B^k strings of k
// symbols (B = sigma + 1 digits: 0 = past the end, 1.. = the symbols in byte order; a gram is its base-B number, so
// numeric order = lexicographic order), weighted by a sampled k-gram histogram of the text.  The code stream of a
// suffix is code(gram at i) code(gram at i + k) ...: comparing streams still equals comparing suffixes, but a gram's
// code length follows the k-th order statistics of the text instead of the symbol frequencies -- DNA + '$' (k = 6):
// 1.9 instead of 2.25 bits per symbol, so 40 key bits cover what 48 did and round 0 sorts in five passes, not six; the
// 97-symbol English-like text (k = 2): six or seven passes instead of eight, and a free top byte for the BWT symbol.
constexpr int GRAM_MIN_K = 4;              // shorter grams see too little context to beat the per-symbol code
constexpr int GRAM_MAX_K = 8;
constexpr int GRAM_MAX_G = 1 << 17;        // table entries (B^k <= this)
constexpr int GRAM_PER_KEY = 16;           // a key takes at most this many grams (degenerate texts: one-bit codes)
constexpr int GRAM_LEN_BITS = 5;           // table entry = code word left-aligned in the upper 27 bits | len, len <= 27
constexpr int GRAM_MAX_LEN = 27;
constexpr uint32_t GRAM_LEN_MASK = (1u << GRAM_LEN_BITS) - 1u;
struct GramCode {
    const uint32_t *tab;   // [G]; nullptr = the per-symbol code (AlphaCode) is in use
    uint32_t k, B, G, pw;  // pw = B^(k-1)
    uint8_t digit[256];    // byte -> digit (bytes that do not occur: 0)
};

// Round-0 parameters derived from the byte histogram of the text -- the single-GPU and the distributed builder
// must key suffixes identically.
struct Round0Plan {
    AlphaCode ac;
    GramCode gram;  // gram.tab != nullptr: keys come from the k-gram code
    uint32_t sigma;
    int b;          // fixed-width code size
    int max_len;    // longest code word
    int bits0;      // key width (multiple of 8, 16..64)
    int k0;         // symbols every key is guaranteed to cover
    int passes0;    // radix passes of round 0
};

// device buffers of the k-gram code: the table (GRAM_MAX_G entries) and the work space of its construction
struct GramScratch {
    uint32_t *tab, *hist;
    uint64_t *cum, *stats;
};

// The complete round-0 plan: the per-symbol code and the key width from the byte histogram; with d_text (the
// single-GPU builder) and an alphabet small enough, the k-gram code, built on the device from a sample of the text,
// whose statistics then decide the key width.  Reads HKCSA_BITS0 (key width), HKCSA_GRAM (0: the per-symbol code
// for every alphabet) and HKCSA_DEBUG_PLAN (prints the gram statistics).
int plan_round0(const uint64_t *h_hist, Round0Plan &p, const uint8_t *d_text = nullptr, uint64_t n = 0,
                const GramScratch *gs = nullptr, cudaStream_t st = nullptr);

// bwt[i] = text[SA[i] - 1] (wrapping to text[n - 1]) by the phased gather of bwt.cu
int bwt_gather(const uint8_t *d_text, const uint32_t *d_sa, uint64_t n, uint8_t *d_bwt, cudaStream_t st);

cudaError_t byte_hist(const uint8_t *d_text, uint64_t n, uint64_t *d_hist, cudaStream_t st);

// 64-bit suffix ids of the distributed build (texts beyond 4 GB, n <= 2^40): id in the low 40 bits, then WIDE_X_BITS
// bits that continue the round-0 key (the code stream behind its 64 bits; 0 when the packer cannot provide them),
// the BWT symbol in the top byte
constexpr int WIDE_ID_BITS = 40;
constexpr int WIDE_X_BITS = 16;
constexpr uint64_t WIDE_ID_MASK = (1ull << WIDE_ID_BITS) - 1ull;
static_assert(WIDE_ID_BITS + WIDE_X_BITS <= 56, "the top byte carries the BWT symbol");

// ---------------------------------------------------------------- round 0: key sources
// The round-0 key of a suffix is the first `bits` bits of its code stream (the last code word truncated).  Every kernel
// that makes or recomputes a key must agree on it bit for bit, so each code writes it once, in a key source:
//   Smem                                shared-memory tile storage;
//   setup(s)                            loads the code's tables, once per CTA (a barrier follows before fill);
//   fill(s, text, n, base, aligned8)    the tile of positions [base, base + PACK_TILE) plus the look-ahead its keys
//                                       reach (aligned8: text + base is 8-byte aligned), barriers included;
//   window(s, j, bits)                  the stream bits from tile position j, left-aligned: key = window >> (64 - bits);
//   at(..., text, n, t, bits)           the key of position t read from global memory (the lazy look-ups).
constexpr int PACK_THREADS = 256;
constexpr int PACK_IPT = 8;
constexpr int PACK_TILE = PACK_THREADS * PACK_IPT;
constexpr int PACK_LOOK = 64;                                   // >= 64 bits of look-ahead (code words >= 1 bit)
constexpr int PACK_VT = PACK_THREADS + PACK_LOOK / PACK_IPT;    // "virtual threads" incl. the look-ahead groups
constexpr int PACK_MAX_LEN = 24;                                // build_alpha_code never exceeds it
constexpr int PACK_STREAM_WORDS = (PACK_TILE + PACK_LOOK) * PACK_MAX_LEN / 32 + 4;

// The per-symbol code (AlphaCode).  The tile's code words go into ONE bit stream in shared memory (each thread owns 8
// consecutive symbols: it sums their code lengths, a block scan gives its bit offset, and it ORs its bits in 32-bit
// pieces); the window of a position is the 64 stream bits at its bit offset -- three shared loads and two funnel
// shifts, whatever the number of symbols the key covers.
struct AlphaKeys {
    AlphaCode code;
    uint32_t max_len;    // longest code word: bounds the stream words a tile touches

    struct Tab {
        uint32_t e[257];     // code << 8 | len by symbol, [256] = past the end
        __device__ __forceinline__ void load(const AlphaCode &c)     // by a block of at least PACK_THREADS threads
        {
            for (uint32_t i = threadIdx.x; i < 257; i += PACK_THREADS) e[i] = (c.code[i] << 8) | c.len[i];
        }
    };
    struct Smem {
        alignas(16) uint16_t off[PACK_TILE];         // bit offset of every tile position in the stream
        uint32_t stream[PACK_STREAM_WORDS];
        Tab tab;
        uint32_t tot[PACK_VT + 24];                  // code bits per group of 8, then their exclusive scan (32 lanes x 9)
        alignas(16) uint16_t off_look[PACK_IPT];     // offsets of a look-ahead group: written, never read
    };

    __device__ __forceinline__ void setup(Smem &s) const
    {
        s.tab.load(code);
        if (threadIdx.x < 24) s.tot[PACK_VT + threadIdx.x] = 0;
    }

    template <typename LenT>
    __device__ __forceinline__ void fill(Smem &s, const uint8_t *__restrict__ text, LenT n, uint64_t base,
                                         bool aligned8) const
    {
        const uint32_t tid = threadIdx.x, lane = tid & 31u;
        // the stream words a tile can touch: (tile + look-ahead) symbols of at most max_len bits
        const uint32_t words = min((uint32_t)PACK_STREAM_WORDS, ((PACK_TILE + PACK_LOOK) * max_len + 31u) / 32u + 4u);
        for (uint32_t i = tid; i < words; i += PACK_THREADS) s.stream[i] = 0;
        __syncthreads();
        const uint8_t *tile = text + base;
        const LenT left = (LenT)(n - base);                         // symbols from the tile's first on
        uint32_t cl[PACK_IPT], cl2[PACK_IPT];
        s.tot[tid] = load8(s.tab, tile, left, tid * PACK_IPT, aligned8, cl);
        if (tid < PACK_LOOK / PACK_IPT)
            s.tot[PACK_THREADS + tid] = load8(s.tab, tile, left, PACK_TILE + tid * PACK_IPT, aligned8, cl2);
        __syncthreads();
        if (tid < 32) {                                             // exclusive scan of the 264 group lengths
            uint32_t v[9], sum = 0;
#pragma unroll
            for (int q = 0; q < 9; ++q) { v[q] = s.tot[lane * 9 + q]; sum += v[q]; }
            uint32_t total;
            uint32_t run = warp_excl_sum(sum, total);
#pragma unroll
            for (int q = 0; q < 9; ++q) { s.tot[lane * 9 + q] = run; run += v[q]; }
        }
        __syncthreads();
        emit8(s.stream, s.off + tid * PACK_IPT, s.tot[tid], cl);
        if (tid < PACK_LOOK / PACK_IPT) emit8(s.stream, s.off_look, s.tot[PACK_THREADS + tid], cl2);
        __syncthreads();
    }

    // x != nullptr: *x = the WIDE_X_BITS stream bits behind the first `bits` (64-bit ids of the distributed build)
    __device__ __forceinline__ uint64_t window(const Smem &s, uint32_t j, int bits, uint16_t *x = nullptr) const
    {
        const uint32_t o = s.off[j];
        const uint32_t wi = o >> 5, sh = o & 31u;
        const uint32_t w0 = s.stream[wi], w1 = s.stream[wi + 1], w2 = s.stream[wi + 2];
        const uint64_t win = ((uint64_t)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);
        if (x) {
            const uint32_t ex = __funnelshift_l(s.stream[wi + 3], w2, sh);
            const uint64_t rest = bits < 64 ? (win << bits) | (((uint64_t)ex << 32) >> (64 - bits)) : ((uint64_t)ex << 32);
            *x = (uint16_t)(rest >> (64 - WIDE_X_BITS));
        }
        return win;
    }

    static __device__ __forceinline__ uint64_t at(const Tab &t, const uint8_t *__restrict__ text, uint64_t n, uint64_t pos,
                                                  int bits)
    {
        uint64_t acc = 0;
        int used = 0;
        for (uint64_t g = pos; used < bits; ++g) {
            const uint32_t c = t.e[g < n ? (uint32_t)text[g] : 256u];
            const int L = c & 0xFFu;
            acc |= ((uint64_t)(c >> 8) << (64 - L)) >> used;    // bits beyond 64 fall off: the last code is truncated
            used += L;
        }
        return acc >> (64 - bits);
    }

private:
    // the 8 symbols from g0 as (code << 8 | len) entries; returns the sum of the lengths
    template <typename LenT>
    static __device__ __forceinline__ uint32_t load8(const Tab &t, const uint8_t *__restrict__ text, LenT n, uint32_t g0,
                                                     bool aligned8, uint32_t cl[PACK_IPT])
    {
        uint32_t total = 0;
        if (aligned8 && g0 + PACK_IPT <= n) {
            const uint2 v = __ldg(reinterpret_cast<const uint2 *>(text + g0));
#pragma unroll
            for (int e = 0; e < PACK_IPT; ++e) {
                const uint32_t c = ((e < 4 ? v.x : v.y) >> (8 * (e & 3))) & 0xFFu;
                cl[e] = t.e[c];
                total += cl[e] & 0xFFu;
            }
        } else {
#pragma unroll
            for (int e = 0; e < PACK_IPT; ++e) {
                const uint32_t g = g0 + e;
                cl[e] = t.e[g < n ? (uint32_t)text[g] : 256u];
                total += cl[e] & 0xFFu;
            }
        }
        return total;
    }

    // ORs the 8 code words into the stream from bit offset `off` (bit 0 = MSB of word 0) and records the bit offset of
    // every symbol
    static __device__ __forceinline__ void emit8(uint32_t *stream, uint16_t *off8, uint32_t off, const uint32_t cl[PACK_IPT])
    {
        uint32_t wi = off >> 5;
        uint32_t nacc = off & 31u;
        uint64_t acc = 0;
        uint32_t o = off;
        uint32_t offs[PACK_IPT];
#pragma unroll
        for (int e = 0; e < PACK_IPT; ++e) {
            const uint32_t L = cl[e] & 0xFFu;
            offs[e] = o;
            o += L;
            acc |= (uint64_t)(cl[e] >> 8) << (64u - nacc - L);     // nacc + L <= 31 + 24
            nacc += L;
            if (nacc >= 32u) {
                atomicOr(&stream[wi++], (uint32_t)(acc >> 32));
                acc <<= 32;
                nacc -= 32u;
            }
        }
        if (nacc) atomicOr(&stream[wi], (uint32_t)(acc >> 32));
        uint4 q;
        q.x = offs[0] | (offs[1] << 16);
        q.y = offs[2] | (offs[3] << 16);
        q.z = offs[4] | (offs[5] << 16);
        q.w = offs[6] | (offs[7] << 16);
        *reinterpret_cast<uint4 *>(off8) = q;
    }
};

// The k-gram code (GramCode).  Per tile: the digits of the tile's symbols (+ the look-ahead a key can reach) into
// shared memory, then the gram at every position by a rolling base-B number and its table entry -- a 4-byte load whose
// hot part (the grams that occur: 16 KB for DNA) stays in L1.  The window of a position ORs the entries at j, j + k,
// j + 2k, ... in at the bits consumed so far (the code word sits left-aligned in the entry: one 64-bit shift per gram).
struct GramKeys {
    GramCode code;

    static constexpr int LOOK = GRAM_PER_KEY * GRAM_MAX_K;      // positions a key can reach beyond its own
    struct Smem {
        uint32_t cl[PACK_TILE + LOOK];                          // table entry of the gram at every position
        alignas(8) uint8_t dig[PACK_TILE + LOOK + 16];          // digits of the symbols
        uint8_t digit[256];
    };

    __device__ __forceinline__ void setup(Smem &s) const { s.digit[threadIdx.x] = code.digit[threadIdx.x]; }

    __device__ __forceinline__ void fill(Smem &s, const uint8_t *__restrict__ text, uint64_t n, uint64_t base,
                                         bool aligned8) const
    {
        constexpr int LOOK_THREADS = LOOK / PACK_IPT;            // 16 threads also take a look-ahead group
        const uint32_t tid = threadIdx.x;
        reinterpret_cast<uint2 *>(s.dig)[tid] = digits8(s.digit, text, n, base + (uint64_t)tid * PACK_IPT, aligned8);
        if (tid < LOOK_THREADS + 2)
            reinterpret_cast<uint2 *>(s.dig)[PACK_THREADS + tid] =
                digits8(s.digit, text, n, base + PACK_TILE + (uint64_t)tid * PACK_IPT, aligned8);
        __syncthreads();
        entries8(s, tid * PACK_IPT);
        if (tid < LOOK_THREADS) entries8(s, PACK_TILE + tid * PACK_IPT);
        __syncthreads();
    }

    __device__ __forceinline__ uint64_t window(const Smem &s, uint32_t j, int bits) const
    {
        uint64_t acc = 0;
        uint32_t used = 0;
        const uint32_t *p = s.cl + j;
        // three grams without a test (3 x 27 bits cannot run past bit 63 of the shift count's range), then until the
        // key is full: most keys of the DNA workload take four
#pragma unroll
        for (int t = 0; t < 3; ++t, p += code.k) {
            const uint32_t c = *p;
            acc |= ((uint64_t)(c & ~GRAM_LEN_MASK) << 32) >> used;
            used += c & GRAM_LEN_MASK;
        }
#pragma unroll 1
        for (int t = 3; t < GRAM_PER_KEY && used < (uint32_t)bits; ++t, p += code.k) {
            const uint32_t c = *p;
            acc |= ((uint64_t)(c & ~GRAM_LEN_MASK) << 32) >> used;
            used += c & GRAM_LEN_MASK;
        }
        return acc;
    }

    __device__ __forceinline__ uint64_t at(const uint8_t *__restrict__ text, uint64_t n, uint64_t pos, int bits) const
    {
        uint64_t acc = 0;
        int used = 0;
        for (int t = 0; t < GRAM_PER_KEY && used < bits; ++t) {
            uint32_t g = 0;
            for (uint32_t q = 0; q < code.k; ++q) {
                const uint64_t p = pos + (uint64_t)t * code.k + q;
                g = g * code.B + (p < n ? (uint32_t)code.digit[text[p]] : 0u);
            }
            const uint32_t c = __ldg(code.tab + g);
            acc |= ((uint64_t)(c & ~GRAM_LEN_MASK) << 32) >> used;      // the code word sits left-aligned in the entry
            used += (int)(c & GRAM_LEN_MASK);
        }
        return acc >> (64 - bits);
    }

    // digits of the 8 symbols from p0, as one 8-byte word (positions past the end: digit 0)
    static __device__ __forceinline__ uint2 digits8(const uint8_t *s_digit, const uint8_t *__restrict__ text, uint64_t n,
                                                    uint64_t p0, bool aligned8)
    {
        uint32_t d[8];
        if (aligned8 && p0 + 8 <= n) {
            const uint2 a = __ldg(reinterpret_cast<const uint2 *>(text + p0));
#pragma unroll
            for (int e = 0; e < 8; ++e) d[e] = s_digit[((e < 4 ? a.x : a.y) >> (8 * (e & 3))) & 0xFFu];
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) d[e] = (p0 + e < n) ? (uint32_t)s_digit[text[p0 + e]] : 0u;
        }
        return make_uint2(d[0] | (d[1] << 8) | (d[2] << 16) | (d[3] << 24), d[4] | (d[5] << 8) | (d[6] << 16) | (d[7] << 24));
    }

    // the grams starting at the 8 positions from j0 (digits in shared memory), by a rolling base-B number
    static __device__ __forceinline__ void roll8(const uint8_t *s_dig, uint32_t j0, uint32_t k, uint32_t B, uint32_t pw,
                                                 uint32_t g[8])
    {
        uint32_t cur = 0;
        for (uint32_t q = 0; q < k; ++q) cur = cur * B + s_dig[j0 + q];
        g[0] = cur;
#pragma unroll
        for (int e = 1; e < 8; ++e) {
            cur = (cur - (uint32_t)s_dig[j0 + e - 1] * pw) * B + s_dig[j0 + e - 1 + k];
            g[e] = cur;
        }
    }

private:
    // table entries of the grams at the 8 positions from j0
    __device__ __forceinline__ void entries8(Smem &s, uint32_t j0) const
    {
        uint32_t g[8], c[8];
        roll8(s.dig, j0, code.k, code.B, code.pw, g);
#pragma unroll
        for (int e = 0; e < 8; ++e) c[e] = __ldg(code.tab + g[e]);
        uint4 *dst = reinterpret_cast<uint4 *>(s.cl + j0);
        dst[0] = make_uint4(c[0], c[1], c[2], c[3]);
        dst[1] = make_uint4(c[4], c[5], c[6], c[7]);
    }
};

// ---------------------------------------------------------------- group-local refinement (suffix_array.cu)
constexpr int GS_MAX = 16;       // groups up to this size are ordered by one thread
constexpr int GS_DEPTH = 64;     // symbols compared beyond the depth the group shares
// keys[j] = (cgrp[j] << 32 | sub-group) with every group of at most GS_MAX elements reordered in place (cidx) by text
// comparison from `depth` on (gram_keys: the groups come from k-gram keys, whose members share far more than `depth`
// symbols -- compared in wider windows); ids64 != nullptr: cidx holds ordinals into ids64 (WIDE_ID_MASK = suffix id,
// then the key extension bits)
cudaError_t group_local_keys(uint32_t *cidx, const uint32_t *cgrp, uint32_t m, const uint8_t *text, uint64_t n,
                             uint64_t depth, bool gram_keys, const uint64_t *ids64, uint64_t *keys, cudaStream_t st);

// ---------------------------------------------------------------- segmented rank update (suffix_array.cu)
// mask = the key bits that were sorted on; carried_out != nullptr: byte j = top byte of sorted key j
__global__ void __launch_bounds__(SEG_THREADS) seg_reduce_kernel(const uint64_t *__restrict__ skey, uint32_t m, uint32_t *__restrict__ agg_head,
                                  uint32_t *__restrict__ agg_keep, uint16_t *__restrict__ flags, uint64_t mask,
                                  uint8_t *__restrict__ carried_out);
__global__ void __launch_bounds__(1024) seg_scan_kernel(uint32_t *__restrict__ agg_head, uint32_t *__restrict__ agg_keep, uint32_t tiles,
                                uint32_t *__restrict__ out_m);
__global__ void __launch_bounds__(SEG_THREADS, 6) seg_apply_kernel(const uint16_t *__restrict__ flags, const uint32_t *__restrict__ sidx,
                                 const uint32_t *__restrict__ pos /* nullptr = identity */, uint32_t m,
                                 const uint32_t *__restrict__ carry_head, const uint32_t *__restrict__ carry_keep,
                                 uint32_t *__restrict__ sa, uint32_t *__restrict__ rank, uint32_t *__restrict__ cpos,
                                 uint32_t *__restrict__ cidx, uint32_t *__restrict__ cgrp, bool write_sa, bool scatter_all,
                                 const uint8_t *__restrict__ text, uint32_t n, uint8_t *__restrict__ bwt);
// the same for round 0 without any rank scatter (pos = identity, nothing placed): the survivors only
void seg_compact0(const uint16_t *flags, const uint32_t *sidx, uint32_t m, const uint32_t *carry_head,
                  const uint32_t *carry_keep, uint32_t *cpos, uint32_t *cidx, uint32_t *cgrp, cudaStream_t st);

}  // namespace hkcsa
