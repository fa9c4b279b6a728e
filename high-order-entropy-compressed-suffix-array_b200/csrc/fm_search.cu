// fm_search.cu -- K4: batched FM-index backward search (count) and locate.
//
// Replaces EnhancedFMIndex.find_range / .rank / .find (reference
// csa/enhanced_fm_index.py:15-40).  occ[c][i] of build_occ (utils/utils.py:
// 26-32) is answered by a rank source: the wavelet tree (WtDev, a rank walk that
// reads one 32-byte block per level), the sampled Occ table (OccDev, occ.cuh) or
// the sliced index of the distributed build (MsDev, multi_slice.cuh); C[] and the
// source's tables live in shared memory.
#include "common.cuh"
#include "multi_slice.cuh"
#include "occ.cuh"
#include "prof.cuh"
#include "radix_sort.cuh"
#include "wavelet.cuh"

namespace hkcsa {

constexpr int COUNT_THREADS = 256;

// the rows a search starts from: a field of the sources over one text, the last start of the sliced index
template <typename Src>
__device__ __forceinline__ typename Src::Row rows_of(const Src &src, const typename Src::Smem &)
{
    return (typename Src::Row)src.n;
}
__device__ __forceinline__ uint64_t rows_of(const MsDev &, const MsSmem &s) { return s.start[s.S]; }

// One lane per pattern.  A warp owns a contiguous chunk of the batch and refills a lane as soon as
// its pattern ends (last symbol consumed or range empty), so ragged lengths (8-64) and early misses do
// not idle the warp: every iteration each busy lane consumes ONE symbol -- both boundaries of the SA
// range take the rank step of the source together (Src: WtDev, OccDev<SHIFT> or MsDev).  find_range
// (csa/enhanced_fm_index.py:21-32) in half-open form:
//   l = 0, r = n;  per symbol from the end: l = C[c] + occ(c, l), r = C[c] + occ(c, r);
//   l >= r -> (-1, -1).  Result (l, r-1).
template <typename Src, int MIN_CTAS, bool PEERS>
__global__ void __launch_bounds__(COUNT_THREADS, MIN_CTAS)
fm_count_kernel(Src src, const uint8_t *__restrict__ pat, const int64_t *__restrict__ off, uint64_t P,
                int64_t *__restrict__ out_lo, int64_t *__restrict__ out_hi, const uint2 *__restrict__ kmer, uint32_t kk,
                PeerOut po)
{
    using Row = typename Src::Row;
    __shared__ typename Src::Smem s;
    src.load(s);
    __syncthreads();
    const Row n = rows_of(src, s);
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t chunk = (P + nwarps - 1) / nwarps;
    uint64_t next = min(P, warp * chunk);
    const uint64_t end = min(P, next + chunk);

    int64_t p = -1;            // pattern owned by this lane, -1 = idle
    int64_t k = 0, b = 0;      // next symbol to consume, first symbol of the pattern
    Row l = 0, r = 0;
    uint32_t ch_next = 0;      // pat[k], loaded one step ahead so the step's rank loads do not wait for it
    while (true) {
        // ---- refill idle lanes with the next patterns of the chunk, in lane order
        const uint32_t idle = __ballot_sync(0xffffffffu, p < 0);
        if (idle) {
            const uint64_t mine = next + __popc(idle & lanemask_lt());
            if (p < 0 && mine < end) {
                p = (int64_t)mine;
                b = off[mine];
                k = off[mine + 1] - 1;
                l = 0;
                r = n;
                // jump table: the SA range of the pattern's last kk symbols was precomputed (by this same
                // search) for every kk-mer over the alphabet; skip those steps.  Its uint2 ranges hold 32-bit rows:
                // the sliced index has none
                if constexpr (sizeof(Row) == 4) if (kmer != nullptr && k - b + 1 >= (int64_t)kk) {
                    uint32_t id = 0;
                    bool known = true;
                    for (uint32_t t = 0; t < kk; ++t) {
                        const uint32_t code = s.code_of_sym[pat[k - kk + 1 + t]];
                        known = known && code != 0xFFFFu;
                        id = id * src.sigma + (known ? code : 0u);
                    }
                    if (known) {
                        const uint2 e2 = __ldg(kmer + id);
                        l = e2.x;
                        r = e2.y;          // l >= r: the kk-mer does not occur
                        k -= kk;
                        if (l >= r) { l = 1; r = 0; k = b - 1; }   // finishes below as a miss
                    }
                }
                if (k >= b) ch_next = pat[k];
            }
            next += __popc(idle);
            if (idle == 0xffffffffu && __ballot_sync(0xffffffffu, p >= 0) == 0) break;
        }
        if (p < 0) continue;
        // ---- one backward-search step (or finish an exhausted / empty pattern)
        bool done = k < b, miss = l >= r;
        if (!done) {
            const uint32_t ch = ch_next;
            if (k > b) ch_next = pat[k - 1];
            const uint32_t code = s.code_of_sym[ch];
            if (code == 0xFFFFu) { miss = true; }          // symbol absent: rank 0, C 0 -> empty range
            else {
                src.rank2(s, code, ch, l, r);
                const Row c0 = s.C[code];
                l += c0;
                r += c0;
                miss = l >= r;
            }
            --k;
            done = miss || k < b;
        }
        if (done) {
            put_range<PEERS>(po, out_lo, out_hi, p, miss ? -1 : (int64_t)l, miss ? -1 : (int64_t)r - 1);
            p = -1;
        }
    }
}

// rows[off[p] + k] = lo[p] + k: one warp per pattern; Row = uint64_t for indexes beyond 2^32 rows
template <typename Row>
__global__ void expand_ranges_kernel(const int64_t *__restrict__ lo, const int64_t *__restrict__ hi,
                                     const int64_t *__restrict__ out_off, uint64_t P, Row *__restrict__ rows)
{
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = lane_id();
    for (uint64_t p = warp; p < P; p += ((uint64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t l = lo[p], h = hi[p];
        if (l < 0) continue;
        const int64_t o = out_off[p];
        for (int64_t k = lane; k <= h - l; k += 32) rows[o + k] = (Row)(l + k);
    }
}

// ---------------------------------------------------------------- results of a sharded batch to every rank
// (lo, hi) of this rank's slice -> packed {lo: low 32 bits, count: high 32 bits} (a miss is lo = 0xFFFFFFFF, count 0)
// stored at [base + p] of the result array of EVERY rank: 8 bytes per pattern instead of the 16 of (lo, hi) as int64.
// A thread packs two patterns and issues one 16-byte store per destination; with a multicast address (NVSwitch)
// ONE multimem.st reaches all ranks.
struct PushDest {
    uint64_t *out[HKCSA_MAX_PEERS];
    uint64_t *mc;            // multicast address of the same array, or nullptr
    uint32_t n;
};
__device__ __forceinline__ uint64_t pack_range(int64_t l, int64_t h)
{
    return l < 0 ? 0x00000000FFFFFFFFull : ((uint64_t)(uint32_t)l | ((uint64_t)(uint32_t)(h - l + 1) << 32));
}
__device__ __forceinline__ void multimem_st16(uint64_t *p, uint64_t a, uint64_t b)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p),
                 "f"(__uint_as_float((uint32_t)a)), "f"(__uint_as_float((uint32_t)(a >> 32))),
                 "f"(__uint_as_float((uint32_t)b)), "f"(__uint_as_float((uint32_t)(b >> 32))) : "memory");
}
__device__ __forceinline__ void multimem_st8(uint64_t *p, uint64_t a)
{
    asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(p),
                 "f"(__uint_as_float((uint32_t)a)), "f"(__uint_as_float((uint32_t)(a >> 32))) : "memory");
}
__global__ void __launch_bounds__(256)
ranges_push_kernel(const int64_t *__restrict__ lo, const int64_t *__restrict__ hi, uint64_t P, uint64_t base, PushDest pd)
{
    const uint64_t first_pair = base >> 1, pairs = ((base + P + 1) >> 1) - first_pair;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t g0 = (first_pair + i) << 1;
        const bool v0 = g0 >= base, v1 = g0 + 1 < base + P;
        const uint64_t a = v0 ? pack_range(lo[g0 - base], hi[g0 - base]) : 0ull;
        const uint64_t b = v1 ? pack_range(lo[g0 + 1 - base], hi[g0 + 1 - base]) : 0ull;
        if (pd.mc) {
            if (v0 && v1) multimem_st16(pd.mc + g0, a, b);
            else if (v0) multimem_st8(pd.mc + g0, a);
            else multimem_st8(pd.mc + g0 + 1, b);
        } else {
            for (uint32_t r = 0; r < pd.n; ++r) {
                if (v0 && v1) *reinterpret_cast<ulonglong2 *>(pd.out[r] + g0) = make_ulonglong2(a, b);
                else if (v0) pd.out[r][g0] = a;
                else pd.out[r][g0 + 1] = b;
            }
        }
    }
}
__global__ void ranges_unpack_kernel(const uint64_t *__restrict__ packed, uint64_t P, int64_t *__restrict__ lo,
                                     int64_t *__restrict__ hi)
{
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t v = packed[p];
        const uint32_t l = (uint32_t)v, c = (uint32_t)(v >> 32);
        const bool miss = c == 0;
        lo[p] = miss ? -1 : (int64_t)l;
        hi[p] = miss ? -1 : (int64_t)l + c - 1;
    }
}

__global__ void gather_u32_kernel(const uint32_t *__restrict__ src, const uint32_t *__restrict__ rows, uint64_t m,
                                  uint32_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < m) out[q] = src[rows[q]];
}

// position of row j: walk LF until a marked row, pos = sample * rate + steps.
// LF(j) = C[c] + occ(c, j) with c = bwt[j], both from one access + rank step of the source.
template <typename Src>
__global__ void __launch_bounds__(256)
locate_rows_kernel(Src src, BitVec marks, const uint32_t *__restrict__ samples, uint32_t rate, uint32_t row0,
                   const uint32_t *__restrict__ rows, uint64_t m, uint32_t *__restrict__ out)
{
    __shared__ typename Src::Smem s;
    __shared__ uint32_t s_c0, s_fix;
    src.load(s);
    __syncthreads();
    if (threadIdx.x == 0) {             // c0 = bwt[row0] = text[n-1]; LF needs fixing iff c0 occurs before row0
        const LfStep t = src.step(s, row0);
        s_c0 = t.code;
        s_fix = t.occ != 0;
    }
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    uint32_t j = rows[q];
    uint32_t steps = 0;
    while (true) {
        uint64_t slot;
        if (marked_slot(marks, j, slot)) {
            out[q] = samples[slot] * rate + steps;
            return;
        }
        // with the exact LF step below a walk meets a marked row within rate-1 steps on every text; the bound only
        // keeps a walk over a corrupt index from spinning
        if (steps >= rate) { out[q] = HKCSA_NO_POSITION; return; }
        const LfStep t = src.step(s, j);
        j = s.C[t.code] + lf_fix(t.occ, t.code, j, s_c0, row0, s_fix);
        ++steps;
    }
}

// The same walk over the sliced index (MsDev, 64-bit global rows): the marks and samples are per slice, so the slice
// of j is looked up once per step and serves both the mark test and the LF step.
__global__ void __launch_bounds__(256)
ms_locate_kernel(MsDev src, const uint64_t *__restrict__ rows, uint64_t m, uint64_t *__restrict__ out)
{
    __shared__ MsSmem s;
    src.load(s);
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const MultiDesc *d = src.d;
    uint64_t j = rows[q];
    uint32_t steps = 0;
    while (true) {
        const uint32_t sl = ms_slice_of(s.start, s.S, j);
        uint64_t slot;
        if (marked_slot(d->marks[sl], (uint32_t)(j - s.start[sl]), slot)) {
            out[q] = (uint64_t)d->samples[sl][slot] * d->rate + steps;
            return;
        }
        // as in locate_rows_kernel: the bound only keeps a walk over a corrupt index from spinning
        if (steps >= d->rate) { out[q] = HKCSA_NO_POSITION64; return; }
        j = src.next(s, src.step(s.start, sl, j), j);
        ++steps;
    }
}

// every kk-mer over the index alphabet, in lexicographic (code) order, as patterns of length kk
__global__ void kmer_patterns_kernel(WtDev wt, uint32_t kk, uint64_t count, uint8_t *__restrict__ pat,
                                     int64_t *__restrict__ off)
{
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id > count) return;
    off[id] = (int64_t)(id * kk);
    if (id == count) return;
    uint64_t v = id;
    for (int t = (int)kk - 1; t >= 0; --t) {
        pat[id * kk + t] = wt.tab->sym_of_code[v % wt.sigma];
        v /= wt.sigma;
    }
}
__global__ void kmer_table_fill_kernel(const int64_t *__restrict__ lo, const int64_t *__restrict__ hi, uint64_t count,
                                       uint2 *__restrict__ table)
{
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= count) return;
    const int64_t l = lo[id], h = hi[id];
    table[id] = (l < 0) ? make_uint2(0u, 0u) : make_uint2((uint32_t)l, (uint32_t)(h + 1));
}

__global__ void symbol_lut_kernel(uint8_t *lut, uint32_t *base, const uint64_t *__restrict__ hist, uint64_t *start)
{
    // single CTA of 256 threads: bucket = byte value, base = exclusive prefix of the histogram
    __shared__ uint64_t s_h[256];
    const uint32_t t = threadIdx.x;
    s_h[t] = hist[t];
    __syncthreads();
    uint64_t pre = 0;
    for (uint32_t c = 0; c < t; ++c) pre += s_h[c];
    lut[t] = (uint8_t)t;
    base[t] = (uint32_t)pre;
    start[t] = pre;
    if (t == 255) start[256] = pre + s_h[255];
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" int hkcsa_count_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint8_t *d_pat,
                                 const int64_t *d_off, uint64_t P, int64_t *d_lo, int64_t *d_hi, void *stream)
{
    return hkcsa_count_batch_kmer(d_blob, h_plan, nullptr, 0, d_pat, d_off, P, d_lo, d_hi, stream);
}

// number of symbols a jump table covers for an alphabet of sigma symbols: the largest k with sigma^k <= 2^21
extern "C" uint32_t hkcsa_kmer_k(uint32_t sigma)
{
    if (sigma < 2) return 0;
    uint32_t k = 0;
    uint64_t v = 1;
    while (k < 16 && v * sigma <= (1ull << 21)) { v *= sigma; ++k; }
    return k;
}
extern "C" uint64_t hkcsa_kmer_entries(uint32_t sigma, uint32_t k)
{
    uint64_t v = 1;
    for (uint32_t t = 0; t < k; ++t) v *= sigma;
    return v;
}
extern "C" size_t hkcsa_kmer_scratch_bytes(uint32_t sigma, uint32_t k)
{
    const uint64_t cnt = hkcsa_kmer_entries(sigma, k);
    Carver c(nullptr);
    c.take<uint8_t>(cnt * k + 16);
    c.take<int64_t>(cnt + 1);
    c.take<int64_t>(cnt);
    c.take<int64_t>(cnt);
    return c.total();
}
// d_table: uint2[sigma^k] = half-open SA range (l, r) of every k-mer (l >= r: does not occur), computed by the
// count kernel itself, so searches that start from the table are bit-identical to full searches.
extern "C" int hkcsa_kmer_table_build(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t k, void *d_table,
                                      void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(h_plan && d_blob && d_table && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(k >= 1 && k <= 16 && h_plan->sigma >= 2, HKCSA_EINVAL, "bad k or alphabet");
    const uint64_t cnt = hkcsa_kmer_entries(h_plan->sigma, k);
    HK_REQUIRE(cnt <= (1ull << 22), HKCSA_EINVAL, "table too large");
    Carver c(d_scratch);
    uint8_t *d_pat = c.take<uint8_t>(cnt * k + 16);
    int64_t *d_off = c.take<int64_t>(cnt + 1);
    int64_t *d_lo = c.take<int64_t>(cnt);
    int64_t *d_hi = c.take<int64_t>(cnt);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "k-mer scratch too small");
    cudaStream_t st = as_stream(stream);
    WtDev wt = make_wt_dev(d_blob, h_plan);
    kmer_patterns_kernel<<<(uint32_t)((cnt + 256) / 256), 256, 0, st>>>(wt, k, cnt, d_pat, d_off);
    HK_LAUNCH_CHECK();
    int rc = hkcsa_count_batch_kmer(d_blob, h_plan, nullptr, 0, d_pat, d_off, cnt, d_lo, d_hi, stream);
    if (rc != HKCSA_OK) return rc;
    kmer_table_fill_kernel<<<(uint32_t)((cnt + 255) / 256), 256, 0, st>>>(d_lo, d_hi, cnt, static_cast<uint2 *>(d_table));
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// The count kernel of rank source Src at MIN_CTAS CTAs per SM (0: no minimum), over a grid of twice the CTAs an SM
// holds (4 when the kernel sets no minimum).
template <typename Src, int MIN_CTAS>
static int count_launch(const Src &src, const uint2 *kmer, uint32_t k, const uint8_t *d_pat, const int64_t *d_off,
                        uint64_t P, int64_t *d_lo, int64_t *d_hi, const PeerOut &po, cudaStream_t st)
{
    const uint64_t per_sm = 2 * (MIN_CTAS ? MIN_CTAS : 4);
    const int blocks = (int)std::min<uint64_t>((P + COUNT_THREADS - 1) / COUNT_THREADS, (uint64_t)num_sms() * per_sm);
    const uint32_t kk = kmer ? k : 0u;
    prof::Scope ps(st, prof::COUNT, 0);
    if (po.n) fm_count_kernel<Src, MIN_CTAS, true><<<blocks, COUNT_THREADS, 0, st>>>(src, d_pat, d_off, P, d_lo, d_hi, kmer, kk, po);
    else fm_count_kernel<Src, MIN_CTAS, false><<<blocks, COUNT_THREADS, 0, st>>>(src, d_pat, d_off, P, d_lo, d_hi, kmer, kk, po);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// count over the sampled Occ table of plan p
static int count_occ(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob, const hkcsa_occ_plan *p,
                     const void *d_kmer_table, uint32_t k, const uint8_t *d_pat, const int64_t *d_off, uint64_t P,
                     int64_t *d_lo, int64_t *d_hi, const PeerOut &po, cudaStream_t st)
{
    HK_REQUIRE(p->n == h_wt->n && p->sigma == h_wt->sigma && p->n >= 1, HKCSA_EINVAL, "occ plan does not match the index");
    const uint2 *kmer = static_cast<const uint2 *>(d_kmer_table);
    return with_occ_source(d_wt_blob, h_wt, d_occ_blob, p, [&](auto occ) {
        using Src = decltype(occ);
        // 4 CTAs/SM (at most 48 registers for layout 1 and for 32 rows per entry, 63 for 64): measured best of 4 / 5 / 6
        // / 8 on the 2.8 GB table (more lanes in flight were slower).  Layout 1: DRAM-resident tables run best at 4 CTAs/SM,
        // tables near the L2 size at 6 (measured: 1.42 vs 1.34 G patterns/s on the 4.8 GB table of the 200 MB text,
        // 3.4 vs 4.0 on the 225 MB DNA table)
        if constexpr (std::is_same_v<Src, OccDev<0>>)
            if (p->blob_bytes <= (1ull << 30)) return count_launch<Src, 6>(occ, kmer, k, d_pat, d_off, P, d_lo, d_hi, po, st);
        return count_launch<Src, 4>(occ, kmer, k, d_pat, d_off, P, d_lo, d_hi, po, st);
    });
}

extern "C" int hkcsa_count_batch_kmer(const void *d_blob, const hkcsa_wt_plan *h_plan, const void *d_kmer_table,
                                      uint32_t k, const uint8_t *d_pat, const int64_t *d_off, uint64_t P,
                                      int64_t *d_lo, int64_t *d_hi, void *stream)
{
    HK_REQUIRE(h_plan && d_blob, HKCSA_EINVAL, "null pointer");
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_off && d_lo && d_hi, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(h_plan->n >= 1, HKCSA_EINVAL, "empty index");
    PeerOut po;
    memset(&po, 0, sizeof(po));
    return count_launch<WtDev, 0>(make_wt_dev(d_blob, h_plan), static_cast<const uint2 *>(d_kmer_table), k, d_pat, d_off,
                                  P, d_lo, d_hi, po, as_stream(stream));
}

extern "C" int hkcsa_count_batch_occ(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob,
                                     const hkcsa_occ_plan *p, const void *d_kmer_table, uint32_t k,
                                     const uint8_t *d_pat, const int64_t *d_off, uint64_t P, int64_t *d_lo,
                                     int64_t *d_hi, void *stream)
{
    HK_REQUIRE(d_wt_blob && h_wt && d_occ_blob && p, HKCSA_EINVAL, "null pointer");
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_off && d_lo && d_hi, HKCSA_EINVAL, "null pointer");
    PeerOut po;
    memset(&po, 0, sizeof(po));
    return count_occ(d_wt_blob, h_wt, d_occ_blob, p, d_kmer_table, k, d_pat, d_off, P, d_lo, d_hi, po, as_stream(stream));
}

extern "C" int hkcsa_count_batch_peers(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob,
                                       const hkcsa_occ_plan *h_occ, const void *d_kmer_table, uint32_t k,
                                       const uint8_t *d_pat, const int64_t *d_off, uint64_t P, uint64_t out_base,
                                       uint32_t n_peers, const uint64_t *h_peer_lo, const uint64_t *h_peer_hi, void *stream)
{
    HK_REQUIRE(d_wt_blob && h_wt && h_peer_lo && h_peer_hi, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n_peers >= 1 && n_peers <= HKCSA_MAX_PEERS, HKCSA_EINVAL, "n_peers must be in [1, HKCSA_MAX_PEERS]");
    HK_REQUIRE((d_occ_blob == nullptr) == (h_occ == nullptr), HKCSA_EINVAL, "occ blob and plan go together");
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_off != nullptr, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(h_wt->n >= 1, HKCSA_EINVAL, "empty index");
    PeerOut po;
    memset(&po, 0, sizeof(po));
    po.n = n_peers;
    po.base = out_base;
    for (uint32_t r = 0; r < n_peers; ++r) {
        HK_REQUIRE(h_peer_lo[r] && h_peer_hi[r], HKCSA_EINVAL, "null peer pointer");
        po.lo[r] = reinterpret_cast<int64_t *>(static_cast<uintptr_t>(h_peer_lo[r]));
        po.hi[r] = reinterpret_cast<int64_t *>(static_cast<uintptr_t>(h_peer_hi[r]));
    }
    cudaStream_t st = as_stream(stream);
    if (d_occ_blob)
        return count_occ(d_wt_blob, h_wt, d_occ_blob, h_occ, d_kmer_table, k, d_pat, d_off, P, nullptr, nullptr, po, st);
    return count_launch<WtDev, 0>(make_wt_dev(d_wt_blob, h_wt), static_cast<const uint2 *>(d_kmer_table), k, d_pat, d_off,
                                  P, nullptr, nullptr, po, st);
}

extern "C" int hkcsa_multi_count_batch(const void *d_desc, const uint8_t *d_pat, const int64_t *d_off, uint64_t P,
                                       int64_t *d_lo, int64_t *d_hi, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_desc && d_off && d_lo && d_hi, HKCSA_EINVAL, "null pointer");
    PeerOut po;
    memset(&po, 0, sizeof(po));
    return count_launch<MsDev, 0>(MsDev{static_cast<const MultiDesc *>(d_desc)}, nullptr, 0, d_pat, d_off, P, d_lo, d_hi,
                                  po, as_stream(stream));
}

extern "C" int hkcsa_expand_ranges(const int64_t *d_lo, const int64_t *d_hi, const int64_t *d_out_off, uint64_t P,
                                   uint32_t *d_rows, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_lo && d_hi && d_out_off, HKCSA_EINVAL, "null pointer");
    const int blocks = (int)std::min<uint64_t>((P * 32 + 255) / 256, (uint64_t)num_sms() * 16);
    expand_ranges_kernel<uint32_t><<<blocks, 256, 0, as_stream(stream)>>>(d_lo, d_hi, d_out_off, P, d_rows);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_expand_ranges64(const int64_t *d_lo, const int64_t *d_hi, const int64_t *d_out_off, uint64_t P,
                                     uint64_t *d_rows, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_lo && d_hi && d_out_off, HKCSA_EINVAL, "null pointer");
    const int blocks = (int)std::min<uint64_t>((P * 32 + 255) / 256, (uint64_t)num_sms() * 16);
    expand_ranges_kernel<uint64_t><<<blocks, 256, 0, as_stream(stream)>>>(d_lo, d_hi, d_out_off, P, d_rows);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_gather_u32(const uint32_t *d_src, const uint32_t *d_rows, uint64_t m, uint32_t *d_out,
                                void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_src && d_rows && d_out, HKCSA_EINVAL, "null pointer");
    gather_u32_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(d_src, d_rows, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

template <typename Src>
static int locate_launch(const Src &src, const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa, uint32_t row0,
                         const uint32_t *d_rows, uint64_t m, uint32_t *d_out_pos, cudaStream_t st)
{
    const uint8_t *sb = static_cast<const uint8_t *>(d_ssa_blob);
    BitVec marks;
    marks.blocks = reinterpret_cast<const RankBlock *>(sb + h_ssa->off_blocks);
    marks.super = reinterpret_cast<const uint64_t *>(sb + h_ssa->off_super);
    marks.len = h_ssa->n;
    prof::Scope ps(st, prof::LOCATE, 0);
    locate_rows_kernel<Src><<<(uint32_t)((m + 255) / 256), 256, 0, st>>>(
        src, marks, reinterpret_cast<const uint32_t *>(sb + h_ssa->off_samples), h_ssa->rate, row0, d_rows, m,
        d_out_pos);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_locate_rows(const void *d_wt_blob, const hkcsa_wt_plan *h_plan, const void *d_ssa_blob,
                                 const hkcsa_ssa_plan *h_ssa, uint32_t row0, const uint32_t *d_rows, uint64_t m,
                                 uint32_t *d_out_pos, void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_wt_blob && h_plan && d_ssa_blob && h_ssa && d_rows && d_out_pos, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(h_ssa->n == h_plan->n, HKCSA_EINVAL, "plans do not match");
    HK_REQUIRE(row0 < h_plan->n, HKCSA_EINVAL, "row0 (the row of suffix 0) out of range");
    return locate_launch(make_wt_dev(d_wt_blob, h_plan), d_ssa_blob, h_ssa, row0, d_rows, m, d_out_pos,
                         as_stream(stream));
}

extern "C" int hkcsa_locate_rows_occ(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob,
                                     const hkcsa_occ_plan *p, const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa,
                                     uint32_t row0, const uint32_t *d_rows, uint64_t m, uint32_t *d_out_pos,
                                     void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_wt_blob && h_wt && d_occ_blob && p && d_ssa_blob && h_ssa && d_rows && d_out_pos, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(p->n == h_wt->n && p->sigma == h_wt->sigma && h_ssa->n == p->n, HKCSA_EINVAL, "plans do not match");
    HK_REQUIRE(row0 < p->n, HKCSA_EINVAL, "row0 (the row of suffix 0) out of range");
    return with_occ_source(d_wt_blob, h_wt, d_occ_blob, p, [&](auto occ) {
        return locate_launch(occ, d_ssa_blob, h_ssa, row0, d_rows, m, d_out_pos, as_stream(stream));
    });
}

extern "C" int hkcsa_multi_locate_rows(const void *d_desc, const uint64_t *d_rows, uint64_t m, uint64_t *d_out_pos,
                                       void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_desc && d_rows && d_out_pos, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    prof::Scope ps(st, prof::LOCATE, 0);
    ms_locate_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, st>>>(MsDev{static_cast<const MultiDesc *>(d_desc)}, d_rows, m,
                                                                 d_out_pos);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_symbol_positions(const uint8_t *d_bwt, uint64_t n, uint32_t *d_pos, uint64_t *d_start,
                                      void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(d_start && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    cudaStream_t st = as_stream(stream);
    Carver c(d_scratch);
    uint64_t *d_hist = c.take<uint64_t>(256);
    uint8_t *d_lut = c.take<uint8_t>(256);
    uint32_t *d_base = c.take<uint32_t>(256);
    uint8_t *d_sorted = c.take<uint8_t>(n + 16);
    SortScratch ss = carve_sort_scratch(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "scratch too small");
    HK_CUDA(hkcsa_byte_hist(d_bwt, n, d_hist, stream) == HKCSA_OK ? cudaSuccess : cudaErrorUnknown);
    symbol_lut_kernel<<<1, 256, 0, st>>>(d_lut, d_base, d_hist, d_start);
    HK_LAUNCH_CHECK();
    if (n == 0) return HKCSA_OK;
    HK_REQUIRE(d_bwt && d_pos, HKCSA_EINVAL, "null pointer");
    HK_CUDA(radix_partition_bytes(d_bwt, d_sorted, d_pos, (uint32_t)n, d_lut, d_base, ss, st));
    return HKCSA_OK;
}

extern "C" size_t hkcsa_symbol_positions_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    c.take<uint64_t>(256);
    c.take<uint8_t>(256);
    c.take<uint32_t>(256);
    c.take<uint8_t>(n + 16);
    carve_sort_scratch(c, n);
    return c.total();
}

extern "C" int hkcsa_ranges_push_peers(const int64_t *d_lo, const int64_t *d_hi, uint64_t P, uint64_t out_base,
                                       uint32_t n_peers, const uint64_t *h_peer_out, uint64_t multicast_out, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_lo && d_hi && (h_peer_out || multicast_out), HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n_peers <= HKCSA_MAX_PEERS && (n_peers >= 1 || multicast_out), HKCSA_EINVAL, "n_peers must be in [1, HKCSA_MAX_PEERS]");
    PushDest pd;
    memset(&pd, 0, sizeof(pd));
    pd.n = n_peers;
    pd.mc = reinterpret_cast<uint64_t *>(static_cast<uintptr_t>(multicast_out));
    for (uint32_t r = 0; r < n_peers && h_peer_out; ++r) {
        HK_REQUIRE((h_peer_out[r] & 15) == 0 && h_peer_out[r], HKCSA_EINVAL, "peer arrays must be 16-byte aligned");
        pd.out[r] = reinterpret_cast<uint64_t *>(static_cast<uintptr_t>(h_peer_out[r]));
    }
    HK_REQUIRE((multicast_out & 15) == 0, HKCSA_EINVAL, "multicast array must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const uint64_t pairs = (P + 2) / 2;
    const int blocks = (int)std::min<uint64_t>((pairs + 255) / 256, (uint64_t)num_sms() * 8);
    // algorithmic bytes: 16 B read, 8 B stored to each of the other ranks over NVLink
    prof::Scope ps(st, prof::OTHER, P * (16 + 8ull * std::max(1u, n_peers)));
    ranges_push_kernel<<<blocks, 256, 0, st>>>(d_lo, d_hi, P, out_base, pd);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_ranges_unpack(const uint64_t *d_packed, uint64_t P, int64_t *d_lo, int64_t *d_hi, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_packed && d_lo && d_hi, HKCSA_EINVAL, "null pointer");
    const int blocks = (int)std::min<uint64_t>((P + 255) / 256, (uint64_t)num_sms() * 8);
    ranges_unpack_kernel<<<blocks, 256, 0, as_stream(stream)>>>(d_packed, P, d_lo, d_hi);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
