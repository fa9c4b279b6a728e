// occ.cuh -- the sampled Occ table (occ_table.cu) as a rank source of the query kernels (fm_search.cu, extract.cu).
//
// Layout 0 (SHIFT = 5 or 6): row r = [2^SHIFT BWT bytes][sigma x u32: occ[code][r << SHIFT]], `stride` bytes apart.
// Layout 1 (SHIFT = 0): per code `stride` 8-byte entries {occ[code][32 r], bitmap of the rows 32 r .. 32 r + 31 that
// hold the code}, then a copy of the BWT at plan.off_bwt.
#pragma once
#include "common.cuh"
#include "wavelet.cuh"

namespace hkcsa {

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

struct OccSmem {
    uint32_t C[260];
    uint16_t code_of_sym[256];
};

template <int SHIFT>
struct OccDev {
    const uint8_t *rows;
    uint64_t stride;          // layout 0: bytes per row; layout 1: entries per code
    const uint8_t *bwt;       // layout 1: the BWT copy at the end of the blob
    const WtTables *tab;      // C[] and the symbol -> code map of the index
    uint32_t sigma;
    uint32_t n;

    using Smem = OccSmem;
    using Row = uint32_t;
    __device__ __forceinline__ void load(OccSmem &s) const
    {
        for (uint32_t i = threadIdx.x; i < 260u; i += blockDim.x) s.C[i] = __ldg(&tab->C[i]);
        for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) s.code_of_sym[i] = __ldg(&tab->code_of_sym[i]);
    }
    __device__ __forceinline__ const uint8_t *row(uint32_t j) const { return rows + (uint64_t)(j >> SHIFT) * stride; }
    __device__ __forceinline__ const uint2 *entries(uint32_t code) const
    {
        return reinterpret_cast<const uint2 *>(rows) + (uint64_t)code * stride;
    }

    // both boundaries of a backward-search step: a <- occ(code, a), b <- occ(code, b).  Layout 0 issues the four
    // loads (two counters, two symbol blocks) together whether or not the boundaries share a row: no divergent paths
    // inside the warp, one memory round trip per step (a shared row is served by the same sectors).
    __device__ __forceinline__ void rank2(const OccSmem &, uint32_t code, uint32_t ch, uint32_t &a, uint32_t &b) const
    {
        if constexpr (SHIFT == 0) {
            const uint2 *e = entries(code);
            const uint2 ea = __ldg(e + (a >> 5));
            const uint2 eb = __ldg(e + (b >> 5));           // the same entry once the range is narrow (merged in L1)
            a = ea.x + __popc(ea.y & ((1u << (a & 31u)) - 1u));
            b = eb.x + __popc(eb.y & ((1u << (b & 31u)) - 1u));
        } else {
            constexpr uint32_t B = 1u << SHIFT;
            const uint32_t ch4 = ch * 0x01010101u;
            const uint8_t *pa = row(a), *pb = row(b);
            const uint32_t base_a = __ldg(reinterpret_cast<const uint32_t *>(pa + B) + code);
            const uint32_t base_b = __ldg(reinterpret_cast<const uint32_t *>(pb + B) + code);
            uint64_t xa[B / 8], xb[B / 8];
            occ_load_row<SHIFT>(pa, xa);
            occ_load_row<SHIFT>(pb, xb);
            a = base_a + __popcll(occ_match_bits<SHIFT>(xa, ch4) & ((1ull << (a & (B - 1))) - 1ull));
            b = base_b + __popcll(occ_match_bits<SHIFT>(xb, ch4) & ((1ull << (b & (B - 1))) - 1ull));
        }
    }

    // the symbol bwt[j] and its count before j: layout 1 reads the BWT byte, then one entry; layout 0 reads both from
    // row j >> SHIFT (two sectors)
    __device__ __forceinline__ LfStep step(const OccSmem &s, uint32_t j) const
    {
        LfStep t;
        if constexpr (SHIFT == 0) {
            t.sym = __ldg(bwt + j);
            t.code = s.code_of_sym[t.sym];
            const uint2 e = __ldg(entries(t.code) + (j >> 5));
            t.occ = e.x + __popc(e.y & ((1u << (j & 31u)) - 1u));
        } else {
            constexpr uint32_t B = 1u << SHIFT;
            const uint8_t *r = row(j);
            const uint32_t o = j & (B - 1);
            uint64_t x[B / 8];
            occ_load_row<SHIFT>(r, x);
            t.sym = __ldg(r + o);                          // same sector as the loads above
            t.code = s.code_of_sym[t.sym];
            const uint32_t base = __ldg(reinterpret_cast<const uint32_t *>(r + B) + t.code);
            t.occ = base + __popcll(occ_match_bits<SHIFT>(x, t.sym * 0x01010101u) & ((1ull << o) - 1ull));
        }
        return t;
    }
    // the plain LF step of extract, as WtDev::next
    __device__ __forceinline__ uint32_t next(const OccSmem &s, const LfStep &t, uint32_t) const
    {
        return s.C[t.code] + t.occ;
    }
};

template <int SHIFT>
static inline OccDev<SHIFT> make_occ_dev(const void *d_blob, const hkcsa_occ_plan *p, const WtTables *tab)
{
    OccDev<SHIFT> o;
    o.rows = static_cast<const uint8_t *>(d_blob);
    o.stride = p->stride;
    o.bwt = o.rows + p->off_bwt;
    o.tab = tab;
    o.sigma = p->sigma;
    o.n = (uint32_t)p->n;
    return o;
}

// f(the Occ table of plan p as the rank source of its layout): OccDev<0> for layout 1, OccDev<5> / OccDev<6> for
// layout 0 with 32 / 64 rows per entry.  C[] and the symbol map come from the wavelet-tree index it belongs to.
template <typename F>
static inline int with_occ_source(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, const void *d_occ_blob,
                                  const hkcsa_occ_plan *p, F &&f)
{
    const WtTables *tab = make_wt_dev(d_wt_blob, h_wt).tab;
    if (p->layout == 1) return f(make_occ_dev<0>(d_occ_blob, p, tab));
    if (p->shift == 5) return f(make_occ_dev<5>(d_occ_blob, p, tab));
    return f(make_occ_dev<6>(d_occ_blob, p, tab));
}

}  // namespace hkcsa
