// extract.cu -- K4c: text back out of the compressed index (the third self-index query next to count and locate).
//
// No reference counterpart: WaveletTree.decompress returns '' (csa/wavelet_tree.py:158-200).  Two kernels:
//
//  * inverse-SA samples: isa[k] = row of the suffix that starts at text position k * rate (k < S = ceil(n / rate)),
//    isa[S] = isa[0].  Derived from the sampled SA alone -- every marked row j has slot r = rank1(marks, j) and
//    samples[r] = SA[j] / rate -- so a loaded index (no text, no full SA) has them too.  The sliced index of the
//    distributed build runs the same kernel once per slice, with the slice's first global row as the row offset.
//  * batched extract: a request [begin, end) is cut at sample boundaries into segments
//    [k * rate, (k + 1) * rate) & [begin, end); each segment is one independent walk that starts at row isa[k + 1]
//    (the suffix just past the segment: its BWT symbol is the segment's last symbol) and emits text[p - 1],
//    text[p - 2], ... by LF steps.  Whole-text extraction is n / rate walks of <= rate steps: a parallel BWT
//    inversion.  Adjacent threads own adjacent segments, so the byte stores of a long range land close together.
//    The LF step comes from a source: the wavelet tree's access + rank descent or the sampled Occ table's (layouts 0
//    and 1), with 32-bit rows and the plain step; or the sliced index (MsDev, multi_slice.cuh), with 64-bit global
//    rows and the exact step, so that it gives the text back on every text.
#include "common.cuh"
#include "multi_slice.cuh"
#include "occ.cuh"
#include "prof.cuh"
#include "wavelet.cuh"

namespace hkcsa {

constexpr int EXT_THREADS = 256;
constexpr int SCAN_THREADS = 1024;

// ---------------------------------------------------------------- inverse-SA samples
// one thread per mark rank block: the marked rows of the block in order, their slots from the block's rank header.
// Row: uint32_t for the index of one text, uint64_t for the sliced index (row_off = the slice's first global row,
// S = the whole text's sample count).
template <typename Row>
__global__ void __launch_bounds__(256)
isa_samples_kernel(BitVec marks, const uint32_t *__restrict__ samples, uint64_t n, uint64_t S, uint64_t row_off,
                   Row *__restrict__ isa)
{
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g * HKCSA_BLOCK_BITS >= n) return;
    const RankBlock b = load_block(marks.blocks + g);
    uint64_t r = marks.super[g / HKCSA_SUPER_BLOCKS] + (uint32_t)(b.w[0] & 0xFFFFFFFFu);
    const uint64_t row0 = g * HKCSA_BLOCK_BITS;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        // payload bit o of the block is bit o + 32 of the 256: word 0 holds payload bits 0-31 in its high half
        uint64_t m = (w == 0) ? (b.w[0] >> 32) : b.w[w];
        const uint64_t base = row0 + (w == 0 ? 0u : 32u + 64u * (w - 1));
        while (m) {
            const uint64_t j = base + (uint64_t)(__ffsll((long long)m) - 1);
            m &= m - 1;
            if (j >= n) break;
            const uint32_t s = samples[r++];
            isa[s] = (Row)(row_off + j);
            if (s == 0) isa[S] = (Row)(row_off + j);   // the walk of the text's last stretch starts at the row of suffix 0
        }
    }
}

// ---------------------------------------------------------------- segments of the requests
// A request clamped to 0 <= b <= e <= n and to its own output slice: whatever the caller passes, the kernel never
// writes outside out[out_off[q] .. out_off[q + 1]).
struct ExtRange {
    uint64_t b, e;
};
__device__ __forceinline__ ExtRange clamp_request(const int64_t *__restrict__ begin, const int64_t *__restrict__ end,
                                               const int64_t *__restrict__ out_off, uint64_t q, uint64_t n)
{
    const int64_t room = max(out_off[q + 1] - out_off[q], (int64_t)0);
    const int64_t b = min(max(begin[q], (int64_t)0), (int64_t)n);
    const int64_t e = min(min(max(end[q], b), (int64_t)n), b + room);
    return ExtRange{(uint64_t)b, (uint64_t)e};
}
__device__ __forceinline__ uint64_t segments_of(const ExtRange &r, uint32_t rate)
{
    return r.e > r.b ? (r.e - 1) / rate - r.b / rate + 1 : 0;
}

// seg_off[q] = segments of the requests before q; three passes (block sums, scan of the block sums, block scans)
__global__ void __launch_bounds__(SCAN_THREADS)
seg_block_sum_kernel(const int64_t *__restrict__ begin, const int64_t *__restrict__ end,
                     const int64_t *__restrict__ out_off, uint64_t R, uint64_t n, uint32_t rate, uint64_t *__restrict__ bsum)
{
    const uint64_t q = (uint64_t)blockIdx.x * SCAN_THREADS + threadIdx.x;
    const uint64_t v = q < R ? segments_of(clamp_request(begin, end, out_off, q, n), rate) : 0;
    uint64_t total;
    block_excl_scan(v, (uint64_t)0, Plus(), total);
    if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// one CTA: exclusive prefix of the block sums in place
__global__ void __launch_bounds__(SCAN_THREADS) seg_scan_sums_kernel(uint64_t *__restrict__ bsum, uint64_t nb)
{
    block_excl_scan_carried(nb, (uint64_t)0, Plus(), [&](uint64_t i) { return bsum[i]; },
                            [&](uint64_t i, uint64_t p) { bsum[i] = p; });
}

__global__ void __launch_bounds__(SCAN_THREADS)
seg_offsets_kernel(const int64_t *__restrict__ begin, const int64_t *__restrict__ end,
                   const int64_t *__restrict__ out_off, uint64_t R, uint64_t n, uint32_t rate,
                   const uint64_t *__restrict__ bsum, uint64_t *__restrict__ seg_off)
{
    const uint64_t q = (uint64_t)blockIdx.x * SCAN_THREADS + threadIdx.x;
    const uint64_t v = q < R ? segments_of(clamp_request(begin, end, out_off, q, n), rate) : 0;
    uint64_t total;
    const uint64_t ex = block_excl_scan(v, (uint64_t)0, Plus(), total) + bsum[blockIdx.x];
    if (q < R) seg_off[q] = ex;
    if (q == R - 1) seg_off[R] = ex + v;
}

// ---------------------------------------------------------------- extract
// Segment t of the batch: request q = the last with seg_off[q] <= t (binary search; a warp's lanes mostly share q
// and read the same offsets), k = its (t - seg_off[q])-th sample block.
__device__ __forceinline__ uint64_t request_of(const uint64_t *__restrict__ seg_off, uint64_t R, uint64_t t)
{
    uint64_t lo = 0, hi = R;                       // seg_off[lo] <= t < seg_off[hi]
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (seg_off[mid] <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

template <typename Row>
struct ExtractArgs {
    const Row *isa;
    uint32_t rate;
    uint64_t n;
    const int64_t *begin, *end, *out_off;
    uint64_t R;
    const uint64_t *seg_off;
    uint8_t *out;
};

// the walks of every segment, grid-strided.  Each step of the source (WtDev, OccDev<SHIFT> or MsDev) gives the symbol
// bwt[j], and its `next` gives LF(j) from that step
template <typename Src>
__global__ void __launch_bounds__(EXT_THREADS) extract_kernel(Src src, ExtractArgs<typename Src::Row> a)
{
    using Row = typename Src::Row;
    __shared__ typename Src::Smem s;
    src.load(s);
    __syncthreads();
    const uint64_t total = a.seg_off[a.R];
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        const uint64_t q = request_of(a.seg_off, a.R, t);
        const ExtRange r = clamp_request(a.begin, a.end, a.out_off, q, a.n);
        const uint64_t k = r.b / a.rate + (t - a.seg_off[q]);
        const uint64_t lo = max(r.b, k * a.rate);
        const uint64_t hi = min(r.e, (k + 1) * a.rate);
        uint64_t p = min((k + 1) * a.rate, a.n);   // the walk starts at the row of the suffix that begins at p
        Row j = __ldg(a.isa + k + 1);
        uint8_t *dst = a.out + a.out_off[q];
        while (p > lo) {
            const auto st = src.step(s, j);
            j = src.next(s, st, j);
            --p;                                   // st.sym = text[p]
            if (p < hi) dst[p - r.b] = (uint8_t)st.sym;
        }
    }
}

// the number of walks is known on the device only: a grid of exactly the resident CTAs strides over them
template <typename K>
int resident_grid(K kernel)
{
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, EXT_THREADS, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    return per_sm * num_sms();
}

}  // namespace hkcsa

using namespace hkcsa;

static int ssa_plan_check(const hkcsa_ssa_plan *p)
{
    HK_REQUIRE(p->rate >= 1, HKCSA_EINVAL, "sampling rate must be >= 1");
    HK_REQUIRE(p->n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    HK_REQUIRE(p->n_samples == (p->n + p->rate - 1) / p->rate, HKCSA_EINVAL,
               "inverse-SA samples need the sampled SA of a whole text (a slice plan samples a part of it)");
    return HKCSA_OK;
}

// the samples of one (slice of a) sampled SA into isa[]: S = the whole text's sample count, row_off = the first row
template <typename Row>
static int isa_samples_launch(const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa, uint64_t S, uint64_t row_off,
                              Row *d_isa, cudaStream_t st)
{
    const uint64_t n = h_ssa->n;
    const uint8_t *sb = static_cast<const uint8_t *>(d_ssa_blob);
    BitVec marks;
    marks.blocks = reinterpret_cast<const RankBlock *>(sb + h_ssa->off_blocks);
    marks.super = reinterpret_cast<const uint64_t *>(sb + h_ssa->off_super);
    marks.len = n;
    const uint64_t nblocks = (n + HKCSA_BLOCK_BITS - 1) / HKCSA_BLOCK_BITS;
    isa_samples_kernel<Row><<<(uint32_t)((nblocks + 255) / 256), 256, 0, st>>>(
        marks, reinterpret_cast<const uint32_t *>(sb + h_ssa->off_samples), n, S, row_off, d_isa);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_isa_samples(const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa, uint32_t *d_isa, void *stream)
{
    HK_REQUIRE(d_ssa_blob && h_ssa && d_isa, HKCSA_EINVAL, "null pointer");
    const int rc = ssa_plan_check(h_ssa);
    if (rc != HKCSA_OK) return rc;
    const uint64_t n = h_ssa->n, S = h_ssa->n_samples;
    if (n == 0) return HKCSA_OK;
    cudaStream_t st = as_stream(stream);
    const uint64_t nblocks = (n + HKCSA_BLOCK_BITS - 1) / HKCSA_BLOCK_BITS;
    // mark blocks and samples read once, S + 1 entries scattered
    prof::Scope ps(st, prof::SSA_BUILD, nblocks * sizeof(RankBlock) + S * 4 + (S + 1) * 4);
    return isa_samples_launch<uint32_t>(d_ssa_blob, h_ssa, S, 0, d_isa, st);
}

extern "C" int hkcsa_multi_isa_samples(uint32_t S, const void *const *d_ssa_blobs,
                                       const hkcsa_ssa_plan *const *h_ssa_plans, const uint64_t *h_starts,
                                       uint64_t *d_isa, void *stream)
{
    HK_REQUIRE(S >= 1 && S <= HKCSA_MAX_SLICES, HKCSA_EINVAL, "1..HKCSA_MAX_SLICES slices");
    HK_REQUIRE(d_ssa_blobs && h_ssa_plans && h_starts && d_isa, HKCSA_EINVAL, "null pointer");
    const uint64_t n = h_starts[S];
    HK_REQUIRE(n <= (1ull << 40), HKCSA_ERANGE, "n exceeds 2^40");
    HK_REQUIRE(h_ssa_plans[0], HKCSA_EINVAL, "null slice");
    const uint32_t rate = h_ssa_plans[0]->rate;
    HK_REQUIRE(rate >= 1, HKCSA_EINVAL, "sampling rate must be >= 1");
    uint64_t samples = 0, blocks = 0;
    for (uint32_t s = 0; s < S; ++s) {
        const hkcsa_ssa_plan *p = h_ssa_plans[s];
        HK_REQUIRE(d_ssa_blobs[s] && p, HKCSA_EINVAL, "null slice");
        HK_REQUIRE(p->rate == rate, HKCSA_EINVAL, "slices sampled at different rates");
        HK_REQUIRE(h_starts[s] <= h_starts[s + 1] && p->n == h_starts[s + 1] - h_starts[s], HKCSA_EINVAL,
                   "slice length != plan length");
        samples += p->n_samples;
        blocks += (p->n + HKCSA_BLOCK_BITS - 1) / HKCSA_BLOCK_BITS;
    }
    const uint64_t total = (n + rate - 1) / rate;
    HK_REQUIRE(total <= (1ull << 32), HKCSA_ERANGE, "ceil(n / rate) exceeds 2^32 (the samples are 32-bit)");
    HK_REQUIRE(samples == total, HKCSA_EINVAL,
               "the slices' samples do not add up to ceil(n / rate) (slices of different builds?)");
    if (n == 0) return HKCSA_OK;
    cudaStream_t st = as_stream(stream);
    // mark blocks and samples read once, S + 1 entries scattered
    prof::Scope ps(st, prof::SSA_BUILD, blocks * sizeof(RankBlock) + total * 4 + (total + 1) * 8);
    for (uint32_t s = 0; s < S; ++s) {
        if (h_ssa_plans[s]->n == 0) continue;
        const int rc = isa_samples_launch<uint64_t>(d_ssa_blobs[s], h_ssa_plans[s], total, h_starts[s], d_isa, st);
        if (rc != HKCSA_OK) return rc;
    }
    return HKCSA_OK;
}

static size_t extract_scratch(uint64_t R, uint64_t **seg_off, uint64_t **bsum, void *base)
{
    Carver c(base);
    *seg_off = c.take<uint64_t>(R + 1);
    *bsum = c.take<uint64_t>((R + SCAN_THREADS - 1) / SCAN_THREADS + 1);
    return c.total();
}

extern "C" size_t hkcsa_extract_scratch_bytes(uint64_t R)
{
    uint64_t *a, *b;
    return extract_scratch(R, &a, &b, nullptr);
}

// Both extract entry points once their own checks passed: the request pointers and the scratch, the segment offsets
// (three scan launches), then the walks over the source's rows.  R >= 1.
template <typename Src>
static int extract_run(Src src, const typename Src::Row *d_isa, uint32_t rate, uint64_t n, const int64_t *d_begin,
                       const int64_t *d_end, const int64_t *d_out_off, uint64_t R, uint8_t *d_out, void *d_scratch,
                       size_t scratch_bytes, cudaStream_t st)
{
    HK_REQUIRE(d_begin && d_end && d_out_off && d_out && d_scratch, HKCSA_EINVAL, "null pointer");
    uint64_t *seg_off, *bsum;
    HK_REQUIRE(extract_scratch(R, &seg_off, &bsum, d_scratch) <= scratch_bytes, HKCSA_ESCRATCH, "extract scratch too small");

    const uint32_t nb = (uint32_t)((R + SCAN_THREADS - 1) / SCAN_THREADS);
    seg_block_sum_kernel<<<nb, SCAN_THREADS, 0, st>>>(d_begin, d_end, d_out_off, R, n, rate, bsum);
    HK_LAUNCH_CHECK();
    seg_scan_sums_kernel<<<1, SCAN_THREADS, 0, st>>>(bsum, nb);
    HK_LAUNCH_CHECK();
    seg_offsets_kernel<<<nb, SCAN_THREADS, 0, st>>>(d_begin, d_end, d_out_off, R, n, rate, bsum, seg_off);
    HK_LAUNCH_CHECK();

    ExtractArgs<typename Src::Row> a{d_isa, rate, n, d_begin, d_end, d_out_off, R, seg_off, d_out};
    prof::Scope ps(st, prof::LOCATE, 0);
    extract_kernel<<<resident_grid(extract_kernel<Src>), EXT_THREADS, 0, st>>>(src, a);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_extract(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const void *d_occ_blob,
                             const hkcsa_occ_plan *h_occ_plan, const uint32_t *d_isa, uint32_t rate,
                             const int64_t *d_begin, const int64_t *d_end, const int64_t *d_out_off, uint64_t R,
                             uint8_t *d_out, void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(d_wt_blob && h_wt_plan && d_isa, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE((d_occ_blob == nullptr) == (h_occ_plan == nullptr), HKCSA_EINVAL, "occ blob and plan go together");
    HK_REQUIRE(rate >= 1, HKCSA_EINVAL, "sampling rate must be >= 1");
    const uint64_t n = h_wt_plan->n;
    HK_REQUIRE(n >= 1 && n <= HKCSA_MAX_N, HKCSA_EINVAL, "empty index or n beyond HKCSA_MAX_N");
    if (h_occ_plan) {
        HK_REQUIRE(h_occ_plan->n == n && h_occ_plan->sigma == h_wt_plan->sigma, HKCSA_EINVAL,
                   "occ plan does not match the index");
        HK_REQUIRE(h_occ_plan->layout == 1 ? h_occ_plan->shift == 5 : (h_occ_plan->shift == 5 || h_occ_plan->shift == 6),
                   HKCSA_EINVAL, "unknown occ table layout");
    }
    if (R == 0) return HKCSA_OK;
    const auto launch = [&](auto src) {
        return extract_run(src, d_isa, rate, n, d_begin, d_end, d_out_off, R, d_out, d_scratch, scratch_bytes,
                           as_stream(stream));
    };
    if (!h_occ_plan) return launch(make_wt_dev(d_wt_blob, h_wt_plan));
    return with_occ_source(d_wt_blob, h_wt_plan, d_occ_blob, h_occ_plan, launch);
}

extern "C" int hkcsa_multi_extract(const void *d_desc, uint64_t n, uint32_t rate, const uint64_t *d_isa,
                                   const int64_t *d_begin, const int64_t *d_end, const int64_t *d_out_off, uint64_t R,
                                   uint8_t *d_out, void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(d_desc && d_isa, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(rate >= 1, HKCSA_EINVAL, "sampling rate must be >= 1");
    HK_REQUIRE(n >= 1, HKCSA_EINVAL, "empty index");
    HK_REQUIRE(n <= (1ull << 40), HKCSA_ERANGE, "n exceeds 2^40");
    if (R == 0) return HKCSA_OK;
    return extract_run(MsDev{static_cast<const MultiDesc *>(d_desc)}, d_isa, rate, n, d_begin, d_end, d_out_off, R,
                       d_out, d_scratch, scratch_bytes, as_stream(stream));
}
