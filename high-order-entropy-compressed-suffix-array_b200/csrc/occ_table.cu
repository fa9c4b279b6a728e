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
//
// This file builds the table; the rank and LF steps that read it are OccDev (occ.cuh), the rank source the query
// kernels of fm_search.cu and extract.cu are instantiated with.
#include "common.cuh"
#include "prof.cuh"
#include "wavelet.cuh"
#include <stdlib.h>

namespace hkcsa {

constexpr int OCC_THREADS = 256;
constexpr int OCC_SUB = 32;           // blocks per sub-chunk of a tile (4 per warp)

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
