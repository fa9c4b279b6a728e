// occ_table.cu -- sampled Occ table: a second rank structure for the query path.
//
// The reference's FM index answers rank(c, i) from a DENSE table occ[c][i] for every symbol and every row
// (build_occ, utils/utils.py:26-32; read by EnhancedFMIndex.rank, csa/enhanced_fm_index.py:34-40) --
// n * sigma integers, impossible beyond a few MB.  This file keeps that table at every B-th row only
// (B = 32 or 64) and stores, next to each kept row, the B BWT symbols the remainder is counted from:
//
//   row r (stride bytes):  [ B BWT bytes of rows r*B .. r*B+B-1 ][ sigma x u32: occ[code][r*B] ]
//   occ(c, i) = row[i / B].count[code(c)] + #{ j < i % B : row[i / B].bwt[j] == c }
//
// One rank = one counter sector + one (B = 32) or two adjacent (B = 64) symbol sectors, independent of the
// alphabet, against one sector PER LEVEL of the wavelet tree (7 levels for the 97-symbol text).  The wavelet
// tree stays the compact index (0.14 B/char/level); this table trades memory (B + 4 sigma bytes per B rows)
// for random-access traffic and is optional.  Ranges are identical by construction (same recurrences).
//
// Layout 1 ("bitmaps") goes one step further: per symbol and per stretch of 32 rows ONE 8-byte entry
//   entry[code][r] = { occ[code][32 r] (u32), bitmap of the rows 32 r .. 32 r + 31 whose BWT symbol is `code` (u32) }
//   occ(c, i) = entry.count + popc(entry.bitmap & ((1 << (i % 32)) - 1))
// so a rank is ONE memory request (the row layout needs the counter sector and the symbol sector; on B200 the
// search is bound by the rate of random requests, not by their size: tools/probes/sector_probe.cu).  Costs
// 8 sigma bytes per 32 rows (24 B per symbol for the 97-symbol text); the blob ends with a copy of the BWT for
// the LF steps of locate.
#include "common.cuh"
#include "prof.cuh"
#include "wavelet.cuh"
#include <stdlib.h>

namespace hkcsa {

constexpr int OCC_THREADS = 256;
constexpr int OCC_SUB = 32;           // blocks per sub-chunk of a tile (4 per warp)

struct OccDev {
    const uint8_t *rows;
    uint64_t stride;      // layout 0: bytes per row; layout 1: entries per code
    const uint8_t *bwt;   // layout 1: the BWT copy at the end of the blob
    uint32_t sigma;
    uint32_t n;
};

// where the symbols / the counter of `code` live inside a row (B = symbols per row)
__device__ __forceinline__ const uint8_t *occ_sym_ptr(const OccDev &o, uint32_t row)
{
    return o.rows + (uint64_t)row * o.stride;
}
__device__ __forceinline__ const uint32_t *occ_cnt_ptr(const uint8_t *sym, uint32_t code, uint32_t B)
{
    return reinterpret_cast<const uint32_t *>(sym + B) + code;
}

// ---------------------------------------------------------------- build
// One CTA per WTL_TILE rows.  gpre[code][tile] (wt_tile_hist + wt_tile_scan) = occurrences before the tile.
template <int SHIFT>
__global__ void __launch_bounds__(OCC_THREADS)
occ_fill_kernel(const uint8_t *__restrict__ bwt, uint64_t n, const WtTables *__restrict__ tab,
                const uint32_t *__restrict__ gpre, uint32_t tiles, uint32_t sigma, uint64_t stride,
                uint8_t *__restrict__ rows, uint64_t nrows)
{
    constexpr uint32_t B = 1u << SHIFT;
    extern __shared__ uint16_t s_cnt[];                 // [OCC_SUB][sigma]
    __shared__ uint32_t s_base[256];
    __shared__ uint8_t s_code[256];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    s_code[tid] = tab->code8_of_sym[tid];
    s_base[tid] = (tid < sigma) ? gpre[(size_t)tid * (tiles + 1) + blockIdx.x] : 0u;
    const uint64_t tile_row0 = (uint64_t)blockIdx.x * (WTL_TILE / B);
    for (uint32_t sub = 0; sub < WTL_TILE / B / OCC_SUB; ++sub) {
        const uint64_t row0 = tile_row0 + (uint64_t)sub * OCC_SUB;
        if (row0 >= nrows) break;
        for (uint32_t i = tid; i < OCC_SUB * sigma; i += OCC_THREADS) s_cnt[i] = 0;
        __syncthreads();
        // ---- per block: copy the symbols, count them per code (match.any: one leader lane adds the group)
        for (uint32_t q = 0; q < OCC_SUB / (OCC_THREADS / 32); ++q) {
            const uint32_t blk = warp * (OCC_SUB / (OCC_THREADS / 32)) + q;
            const uint64_t row = row0 + blk;
            if (row >= nrows) break;
            uint8_t *dst = rows + row * stride;
#pragma unroll
            for (uint32_t r = 0; r < B / 32; ++r) {
                const uint64_t pos = row * B + r * 32u + lane;
                const bool valid = pos < n;
                const uint32_t ch = valid ? (uint32_t)bwt[pos] : 0u;
                dst[r * 32u + lane] = (uint8_t)ch;
                const uint32_t code = valid ? (uint32_t)s_code[ch] : 256u + lane;
                const uint32_t peers = __match_any_sync(0xffffffffu, code);
                if (valid && lane == (uint32_t)(__ffs(peers) - 1)) s_cnt[blk * sigma + code] += (uint16_t)__popc(peers);
                __syncwarp();
            }
        }
        __syncthreads();
        // ---- per code: running count over the blocks of the sub-chunk -> the rows' counters
        if (tid < sigma) {
            uint32_t run = s_base[tid];
            for (uint32_t blk = 0; blk < OCC_SUB; ++blk) {
                const uint64_t row = row0 + blk;
                if (row >= nrows) break;
                reinterpret_cast<uint32_t *>(rows + row * stride + B)[tid] = run;
                run += s_cnt[blk * sigma + tid];
            }
            s_base[tid] = run;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- rank
// bit j of the result = (byte j of the block == ch), for the 2^SHIFT bytes held in x[]
template <int SHIFT>
__device__ __forceinline__ uint64_t occ_match_bits(const uint64_t (&x)[(1 << SHIFT) / 8], uint32_t ch4)
{
    uint64_t bits = 0;
#pragma unroll
    for (int v = 0; v < (1 << SHIFT) / 8; ++v) {
        const uint32_t lo = __vcmpeq4((uint32_t)x[v], ch4) & 0x01010101u;           // 1 per equal byte
        const uint32_t hi = __vcmpeq4((uint32_t)(x[v] >> 32), ch4) & 0x01010101u;
        const uint32_t byte = ((lo * 0x01020408u) >> 24) | (((hi * 0x01020408u) >> 24) << 4);   // byte i -> bit i
        bits |= (uint64_t)byte << (8 * v);
    }
    return bits;
}
// the row's symbols: one 256-bit load per 32 bytes (LDG.E.256).  (L1::no_allocate was measured: same L2 and DRAM
// traffic, 60 % slower on the 2.8 GB table -- fewer requests in flight on that path.)
template <int SHIFT>
__device__ __forceinline__ void occ_load_row(const uint8_t *sym, uint64_t (&x)[(1 << SHIFT) / 8])
{
#pragma unroll
    for (int v = 0; v < (1 << SHIFT) / 32; ++v) ld_nc_256(sym + 32 * v, x[4 * v], x[4 * v + 1], x[4 * v + 2], x[4 * v + 3]);
}
// occurrences of `ch` among the first t bytes (t < 2^SHIFT) of the row whose symbols start at `sym`
template <int SHIFT>
__device__ __forceinline__ uint32_t occ_count(const uint8_t *sym, uint32_t ch4, uint32_t t)
{
    uint64_t x[(1 << SHIFT) / 8];
    occ_load_row<SHIFT>(sym, x);
    return __popcll(occ_match_bits<SHIFT>(x, ch4) & ((1ull << t) - 1ull));
}

// both boundaries of a backward-search step: a <- occ(code, a), b <- occ(code, b).  The four loads (two
// counters, two symbol blocks) are issued together whether or not the boundaries share a row: no divergent
// paths inside the warp, one memory round trip per step (a shared row is served by the same sectors).
template <int SHIFT>
__device__ __forceinline__ void occ_rank2(const OccDev &o, uint32_t code, uint32_t ch, uint32_t &a, uint32_t &b)
{
    constexpr uint32_t B = 1u << SHIFT;
    const uint32_t ch4 = ch * 0x01010101u;
    const uint8_t *pa = occ_sym_ptr(o, a >> SHIFT);
    const uint8_t *pb = occ_sym_ptr(o, b >> SHIFT);
    const uint32_t base_a = __ldg(occ_cnt_ptr(pa, code, B));
    const uint32_t base_b = __ldg(occ_cnt_ptr(pb, code, B));
    uint64_t xa[B / 8], xb[B / 8];
    occ_load_row<SHIFT>(pa, xa);
    occ_load_row<SHIFT>(pb, xb);
    a = base_a + __popcll(occ_match_bits<SHIFT>(xa, ch4) & ((1ull << (a & (B - 1))) - 1ull));
    b = base_b + __popcll(occ_match_bits<SHIFT>(xb, ch4) & ((1ull << (b & (B - 1))) - 1ull));
}

// ---------------------------------------------------------------- layout 1: per-symbol bitmaps
__global__ void __launch_bounds__(OCC_THREADS)
occ_bitmap_fill_kernel(const uint8_t *__restrict__ bwt, uint64_t n, const WtTables *__restrict__ tab,
                       const uint32_t *__restrict__ gpre, uint32_t tiles, uint32_t sigma, uint64_t per_code,
                       uint2 *__restrict__ entries, uint64_t nrows)
{
    extern __shared__ uint32_t s_mask[];                // [OCC_SUB][sigma]
    __shared__ uint32_t s_base[256];
    __shared__ uint8_t s_code[256];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    s_code[tid] = tab->code8_of_sym[tid];
    s_base[tid] = (tid < sigma) ? gpre[(size_t)tid * (tiles + 1) + blockIdx.x] : 0u;
    const uint64_t tile_row0 = (uint64_t)blockIdx.x * (WTL_TILE / 32);
    for (uint32_t sub = 0; sub < WTL_TILE / 32 / OCC_SUB; ++sub) {
        const uint64_t row0 = tile_row0 + (uint64_t)sub * OCC_SUB;
        if (row0 >= nrows) break;
        for (uint32_t i = tid; i < OCC_SUB * sigma; i += OCC_THREADS) s_mask[i] = 0;
        __syncthreads();
        for (uint32_t q = 0; q < OCC_SUB / (OCC_THREADS / 32); ++q) {
            const uint32_t blk = warp * (OCC_SUB / (OCC_THREADS / 32)) + q;
            const uint64_t row = row0 + blk;
            if (row >= nrows) break;
            const uint64_t pos = row * 32u + lane;
            const bool valid = pos < n;
            const uint32_t code = valid ? (uint32_t)s_code[bwt[pos]] : 256u + lane;
            const uint32_t peers = __match_any_sync(0xffffffffu, code);      // the lanes = the rows holding `code`
            if (valid && lane == (uint32_t)(__ffs(peers) - 1)) s_mask[blk * sigma + code] = peers;
        }
        __syncthreads();
        // one warp per code: lane l owns row row0 + l, the running count is a warp scan of the popcounts, and the
        // 32 entries of the code go out as one contiguous 256-byte store
        static_assert(OCC_SUB == 32, "one lane per row of the sub-chunk");
        for (uint32_t c = warp; c < sigma; c += OCC_THREADS / 32) {
            const uint64_t row = row0 + lane;
            const uint32_t m = (row < nrows) ? s_mask[lane * sigma + c] : 0u;
            uint32_t total;
            const uint32_t ex = warp_excl_sum(__popc(m), total);
            const uint32_t base = s_base[c];
            if (row < nrows) entries[(uint64_t)c * per_code + row] = make_uint2(base + ex, m);
            __syncwarp();
            if (lane == 0) s_base[c] = base + total;
        }
        __syncthreads();
    }
}

// SHIFT = 0 selects the bitmap layout in the search kernels
template <>
__device__ __forceinline__ void occ_rank2<0>(const OccDev &o, uint32_t code, uint32_t ch, uint32_t &a, uint32_t &b)
{
    const uint2 *e = reinterpret_cast<const uint2 *>(o.rows) + (uint64_t)code * o.stride;
    const uint2 ea = __ldg(e + (a >> 5));
    const uint2 eb = __ldg(e + (b >> 5));           // the same entry once the range is narrow (merged in L1)
    a = ea.x + __popc(ea.y & ((1u << (a & 31u)) - 1u));
    b = eb.x + __popc(eb.y & ((1u << (b & 31u)) - 1u));
}

// Same search as fm_count_kernel (fm_search.cu): one lane per pattern, lanes refilled as patterns end;
// find_range (csa/enhanced_fm_index.py:21-32) in half-open form.  Only the rank primitive differs.
template <int SHIFT, int MIN_CTAS, bool PEERS>
__global__ void __launch_bounds__(OCC_THREADS, MIN_CTAS)
fm_count_occ_kernel(OccDev occ, const WtTables *__restrict__ tab, const uint8_t *__restrict__ pat,
                    const int64_t *__restrict__ off, uint64_t P, int64_t *__restrict__ out_lo,
                    int64_t *__restrict__ out_hi, const uint2 *__restrict__ kmer, uint32_t kk, PeerOut po)
{
    __shared__ uint32_t s_C[260];
    __shared__ uint16_t s_code[256];
    for (uint32_t i = threadIdx.x; i < 260u; i += blockDim.x) s_C[i] = tab->C[i];
    for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) s_code[i] = tab->code_of_sym[i];
    __syncthreads();
    const uint32_t n = occ.n;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t chunk = (P + nwarps - 1) / nwarps;
    uint64_t next = min(P, warp * chunk);
    const uint64_t end = min(P, next + chunk);

    int64_t p = -1;
    int64_t k = 0, b = 0;
    uint32_t l = 0, r = 0;
    uint32_t ch_next = 0;      // pat[k], loaded one step ahead so the step's rank loads do not wait for it
    while (true) {
        const uint32_t idle = __ballot_sync(0xffffffffu, p < 0);
        if (idle) {
            const uint64_t mine = next + __popc(idle & lanemask_lt());
            if (p < 0 && mine < end) {
                p = (int64_t)mine;
                b = off[mine];
                k = off[mine + 1] - 1;
                l = 0;
                r = n;
                if (kmer != nullptr && k - b + 1 >= (int64_t)kk) {
                    uint32_t id = 0;
                    bool known = true;
                    for (uint32_t t = 0; t < kk; ++t) {
                        const uint32_t code = s_code[pat[k - kk + 1 + t]];
                        known = known && code != 0xFFFFu;
                        id = id * occ.sigma + (known ? code : 0u);
                    }
                    if (known) {
                        const uint2 e2 = __ldg(kmer + id);
                        l = e2.x;
                        r = e2.y;
                        k -= kk;
                        if (l >= r) { l = 1; r = 0; k = b - 1; }
                    }
                }
                if (k >= b) ch_next = pat[k];
            }
            next += __popc(idle);
            if (idle == 0xffffffffu && __ballot_sync(0xffffffffu, p >= 0) == 0) break;
        }
        if (p < 0) continue;
        bool done = k < b, miss = l >= r;
        if (!done) {
            const uint32_t ch = ch_next;
            if (k > b) ch_next = pat[k - 1];
            const uint32_t code = s_code[ch];
            if (code == 0xFFFFu) { miss = true; }
            else {
                occ_rank2<SHIFT>(occ, code, ch, l, r);
                const uint32_t c0 = s_C[code];
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

// occ(bwt[j], j) from the Occ table, and the symbol's code
template <int SHIFT>
__device__ __forceinline__ uint32_t occ_step(const OccDev &occ, const uint16_t *s_code, uint32_t j, uint32_t &code)
{
    constexpr uint32_t B = 1u << SHIFT;
    if (SHIFT == 0) {
        const uint32_t ch = __ldg(occ.bwt + j);
        code = s_code[ch];
        const uint2 e = __ldg(reinterpret_cast<const uint2 *>(occ.rows) + (uint64_t)code * occ.stride + (j >> 5));
        return e.x + __popc(e.y & ((1u << (j & 31u)) - 1u));
    } else {
        const uint32_t t = j & (B - 1);
        const uint8_t *row = occ_sym_ptr(occ, j >> SHIFT);
        const uint32_t ch = __ldg(row + t);
        code = s_code[ch];
        return __ldg(occ_cnt_ptr(row, code, B)) + occ_count<(SHIFT ? SHIFT : 5)>(row, ch * 0x01010101u, t);
    }
}

// position of row j: LF walk until a marked row (locate_rows_kernel of fm_search.cu with the LF step read from
// the Occ table: the symbol bwt[j] and its count before j come from the same row -- two sectors per step)
template <int SHIFT>
__global__ void __launch_bounds__(256)
locate_rows_occ_kernel(OccDev occ, const WtTables *__restrict__ tab, BitVec marks, const uint32_t *__restrict__ samples,
                       uint32_t rate, uint32_t row0, const uint32_t *__restrict__ rows, uint64_t m,
                       uint32_t *__restrict__ out)
{
    __shared__ uint32_t s_C[260];
    __shared__ uint16_t s_code[256];
    __shared__ uint32_t s_c0, s_fix;
    for (uint32_t i = threadIdx.x; i < 260u; i += blockDim.x) s_C[i] = tab->C[i];
    for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) s_code[i] = tab->code_of_sym[i];
    __syncthreads();
    if (threadIdx.x == 0) {             // c0 = bwt[row0]; the LF step needs lf_fix iff c0 occurs before row0
        uint32_t c0;
        s_fix = occ_step<SHIFT>(occ, s_code, row0, c0) != 0;
        s_c0 = c0;
    }
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    uint32_t j = rows[q];
    uint32_t steps = 0;
    while (true) {
        const uint64_t g = j / HKCSA_BLOCK_BITS;
        const uint32_t o = j - (uint32_t)g * HKCSA_BLOCK_BITS;
        const RankBlock b = load_block(marks.blocks + g);
        if (block_bit(b, o)) {
            const uint64_t r = marks.super[g / HKCSA_SUPER_BLOCKS] + (uint32_t)(b.w[0] & 0xFFFFFFFFu) + block_rank(b, o);
            out[q] = samples[r] * rate + steps;
            return;
        }
        if (steps >= rate) { out[q] = HKCSA_NO_POSITION; return; }   // corrupt index only: see locate_rows_kernel
        uint32_t code;
        const uint32_t cnt = occ_step<SHIFT>(occ, s_code, j, code);
        j = s_C[code] + lf_fix(cnt, code, j, s_c0, row0, s_fix);
        ++steps;
    }
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" int hkcsa_occ_plan_make(uint64_t n, uint32_t sigma, uint32_t shift, uint32_t layout, hkcsa_occ_plan *p)
{
    HK_REQUIRE(p != nullptr, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(shift == 5 || shift == 6, HKCSA_EINVAL, "shift must be 5 (32 rows per entry) or 6 (64)");
    HK_REQUIRE(layout == 0 || (layout == 1 && shift == 5), HKCSA_EINVAL, "layout 1 (per-symbol bitmaps) has 32 rows per entry");
    HK_REQUIRE(sigma >= 1 && sigma <= 256, HKCSA_EINVAL, "bad alphabet size");
    HK_REQUIRE(n >= 1 && n <= HKCSA_MAX_N, HKCSA_ERANGE, "n out of range");
    memset(p, 0, sizeof(*p));
    p->n = n;
    p->sigma = sigma;
    p->shift = shift;
    p->rows = (n >> shift) + 1;
    p->layout = layout;
    if (layout == 1) {
        p->stride = align_up(p->rows, 4);                                  // entries per code (32-byte multiples)
        p->off_bwt = align_up((uint64_t)sigma * p->stride * 8, 256);
        p->blob_bytes = align_up(p->off_bwt + n, 256);
    } else {
        p->stride = align_up(((size_t)1 << shift) + 4 * (size_t)sigma, 32);
        p->blob_bytes = align_up(p->rows * p->stride, 256);
    }
    const uint64_t tiles = (n + WTL_TILE - 1) / WTL_TILE;
    Carver c(nullptr);
    c.take<uint32_t>((uint64_t)sigma * (tiles + 2));
    p->scratch_bytes = c.total();
    return HKCSA_OK;
}

extern "C" int hkcsa_occ_build(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const uint8_t *d_bwt,
                               const hkcsa_occ_plan *p, void *d_blob, void *d_scratch, size_t scratch_bytes,
                               void *stream)
{
    HK_REQUIRE(d_wt_blob && h_wt && d_bwt && p && d_blob && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(p->n == h_wt->n && p->sigma == h_wt->sigma, HKCSA_EINVAL, "occ plan does not match the index");
    HK_REQUIRE(scratch_bytes >= p->scratch_bytes, HKCSA_ESCRATCH, "occ scratch too small");
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_blob) & 63) == 0, HKCSA_EINVAL, "d_blob must be 64-byte aligned");
    cudaStream_t st = as_stream(stream);
    const uint64_t n = p->n;
    const uint32_t tiles = (uint32_t)((n + WTL_TILE - 1) / WTL_TILE);
    const WtTables *d_tab = reinterpret_cast<const WtTables *>(static_cast<const uint8_t *>(d_wt_blob) + h_wt->off_tables);
    Carver c(d_scratch);
    uint32_t *d_gcnt = c.take<uint32_t>((uint64_t)p->sigma * (tiles + 2));
    prof::Scope ps(st, prof::OTHER, n + p->rows * p->stride);
    wt_tile_hist_kernel<<<tiles, WTL_THREADS, 0, st>>>(d_bwt, n, d_tab, p->sigma, tiles, d_gcnt);
    HK_LAUNCH_CHECK();
    wt_tile_scan_kernel<<<p->sigma, 1024, 0, st>>>(d_gcnt, tiles);
    HK_LAUNCH_CHECK();
    // the row of position n exists even when n is a multiple of the tile: one more CTA then reads the totals
    const uint32_t grid = (uint32_t)(n / WTL_TILE) + 1;
    uint8_t *rows = static_cast<uint8_t *>(d_blob);
    if (p->layout == 1) {
        const size_t smem1 = (size_t)OCC_SUB * p->sigma * sizeof(uint32_t);
        occ_bitmap_fill_kernel<<<grid, OCC_THREADS, smem1, st>>>(d_bwt, n, d_tab, d_gcnt, tiles, p->sigma, p->stride,
                                                                 reinterpret_cast<uint2 *>(rows), p->rows);
        HK_LAUNCH_CHECK();
        HK_CUDA(cudaMemcpyAsync(rows + p->off_bwt, d_bwt, n, cudaMemcpyDeviceToDevice, st));
        return HKCSA_OK;
    }
    const size_t smem = (size_t)OCC_SUB * p->sigma * sizeof(uint16_t);
    if (p->shift == 5)
        occ_fill_kernel<5><<<grid, OCC_THREADS, smem, st>>>(d_bwt, n, d_tab, d_gcnt, tiles, p->sigma, p->stride, rows, p->rows);
    else
        occ_fill_kernel<6><<<grid, OCC_THREADS, smem, st>>>(d_bwt, n, d_tab, d_gcnt, tiles, p->sigma, p->stride, rows, p->rows);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

static int count_occ_launch(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob,
                            const hkcsa_occ_plan *p, const void *d_kmer_table, uint32_t k, const uint8_t *d_pat,
                            const int64_t *d_off, uint64_t P, int64_t *d_lo, int64_t *d_hi, const PeerOut &po,
                            cudaStream_t st)
{
    HK_REQUIRE(p->n == h_wt->n && p->sigma == h_wt->sigma && p->n >= 1, HKCSA_EINVAL, "occ plan does not match the index");
    const WtTables *d_tab = reinterpret_cast<const WtTables *>(static_cast<const uint8_t *>(d_wt_blob) + h_wt->off_tables);
    OccDev occ;
    occ.rows = static_cast<const uint8_t *>(d_occ_blob);
    occ.stride = p->stride;
    occ.bwt = occ.rows + p->off_bwt;
    occ.sigma = p->sigma;
    occ.n = (uint32_t)p->n;
    const uint2 *kmer = static_cast<const uint2 *>(d_kmer_table);
    const uint32_t kk = kmer ? k : 0u;
    prof::Scope ps(st, prof::COUNT, 0);
    // 4 CTAs/SM (53 registers): measured best of 4 / 5 / 6 / 8 on the 2.8 GB table (more lanes in flight were slower)
    const int blocks = (int)std::min<uint64_t>((P + OCC_THREADS - 1) / OCC_THREADS, (uint64_t)num_sms() * 8);
#define OCC_COUNT(SH, MC, GRID)                                                                                         \
    do {                                                                                                                \
        if (po.n) fm_count_occ_kernel<SH, MC, true><<<GRID, OCC_THREADS, 0, st>>>(occ, d_tab, d_pat, d_off, P, d_lo, d_hi, kmer, kk, po);  \
        else fm_count_occ_kernel<SH, MC, false><<<GRID, OCC_THREADS, 0, st>>>(occ, d_tab, d_pat, d_off, P, d_lo, d_hi, kmer, kk, po);      \
    } while (0)
    if (p->layout == 1) {
        // lanes in flight: DRAM-resident tables run best at 4 CTAs/SM, tables near the L2 size at 6 (measured:
        // 1.42 vs 1.34 G patterns/s on the 4.8 GB table of the 200 MB text, 3.4 vs 4.0 on the 225 MB DNA table)
        const int ctas = (p->blob_bytes > (1ull << 30)) ? 4 : 6;
        const int blocks1 = (int)std::min<uint64_t>((P + OCC_THREADS - 1) / OCC_THREADS, (uint64_t)num_sms() * 2 * ctas);
        if (ctas == 6) OCC_COUNT(0, 6, blocks1);
        else OCC_COUNT(0, 4, blocks1);
    } else if (p->shift == 5) {
        OCC_COUNT(5, 4, blocks);
    } else {
        OCC_COUNT(6, 4, blocks);
    }
#undef OCC_COUNT
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
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
    return count_occ_launch(d_wt_blob, h_wt, d_occ_blob, p, d_kmer_table, k, d_pat, d_off, P, d_lo, d_hi, po, as_stream(stream));
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
        return count_occ_launch(d_wt_blob, h_wt, d_occ_blob, h_occ, d_kmer_table, k, d_pat, d_off, P, nullptr, nullptr, po, st);
    return count_wt_launch(make_wt_dev(d_wt_blob, h_wt), static_cast<const uint2 *>(d_kmer_table), k, d_pat, d_off, P,
                           nullptr, nullptr, po, st);
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
    cudaStream_t st = as_stream(stream);
    const WtTables *d_tab = reinterpret_cast<const WtTables *>(static_cast<const uint8_t *>(d_wt_blob) + h_wt->off_tables);
    OccDev occ;
    occ.rows = static_cast<const uint8_t *>(d_occ_blob);
    occ.stride = p->stride;
    occ.bwt = occ.rows + p->off_bwt;
    occ.sigma = p->sigma;
    occ.n = (uint32_t)p->n;
    const uint8_t *sb = static_cast<const uint8_t *>(d_ssa_blob);
    BitVec marks;
    marks.blocks = reinterpret_cast<const RankBlock *>(sb + h_ssa->off_blocks);
    marks.super = reinterpret_cast<const uint64_t *>(sb + h_ssa->off_super);
    marks.len = h_ssa->n;
    const uint32_t *samples = reinterpret_cast<const uint32_t *>(sb + h_ssa->off_samples);
    const uint32_t grid = (uint32_t)((m + 255) / 256);
    prof::Scope ps(st, prof::LOCATE, 0);
    if (p->layout == 1)
        locate_rows_occ_kernel<0><<<grid, 256, 0, st>>>(occ, d_tab, marks, samples, h_ssa->rate, row0, d_rows, m,
                                                            d_out_pos);
    else if (p->shift == 5)
        locate_rows_occ_kernel<5><<<grid, 256, 0, st>>>(occ, d_tab, marks, samples, h_ssa->rate, row0, d_rows, m,
                                                            d_out_pos);
    else
        locate_rows_occ_kernel<6><<<grid, 256, 0, st>>>(occ, d_tab, marks, samples, h_ssa->rate, row0, d_rows, m,
                                                            d_out_pos);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
