// multi_slice.cuh -- the sliced index of the distributed build: its descriptor (built by multi_slice.cu) and MsDev, the
// rank source that count and locate (fm_search.cu) and extract (extract.cu) run on.
#pragma once
#include "common.cuh"
#include "wavelet.cuh"

namespace hkcsa {

struct MultiDesc {
    WtDev slice[HKCSA_MAX_SLICES];
    BitVec marks[HKCSA_MAX_SLICES];
    const uint32_t *samples[HKCSA_MAX_SLICES];
    uint64_t start[HKCSA_MAX_SLICES + 1];
    uint64_t cum[HKCSA_MAX_SLICES + 1][256];   // occurrences of byte c in slices < s  ([S] = total)
    uint64_t C[256];                           // symbols of the whole text smaller than byte c
    uint32_t S;
    uint32_t rate;                             // 0 = no sampled SA
    uint64_t n;
    uint64_t row0;                             // global row of suffix 0 (UINT64_MAX: no sampled SA)
};

// the slice holding global row i; `start` is the descriptor's or a shared-memory copy of it
__device__ __forceinline__ uint32_t ms_slice_of(const uint64_t *start, uint32_t S, uint64_t i)
{
    uint32_t s = 0;
    for (uint32_t k = 1; k < S; ++k) s += (i >= start[k]) ? 1u : 0u;
    return s;
}

// The sliced index as a rank source, on 64-bit global rows.  Slice s covers rows [start[s], start[s+1]) and has its
// own wavelet tree, whose codes are its own: the source's codes are the bytes, absent ones 0xFFFF.  occ(c, i) =
// cum[s][c] (occurrences of c in earlier slices) + the rank of c inside the slice s holding i; the descents read the
// slice's node tables from global memory on the read-only path.  The starts, C[], cum[][] (16 KB at 8 slices) and the
// byte map are in shared memory; c0 and fix of the exact LF step are read once per CTA from row0.
struct MsSmem {
    uint64_t start[HKCSA_MAX_SLICES + 1];
    uint64_t cum[HKCSA_MAX_SLICES][256];
    uint64_t C[256];
    uint64_t row0;
    uint16_t code_of_sym[256];
    uint32_t S, c0, fix;
};
struct MsStep {
    uint32_t slice, sym, occ;             // occ: occurrences of sym in the slice before j
};
struct MsDev {
    const MultiDesc *d;

    using Smem = MsSmem;
    using Row = uint64_t;
    __device__ __forceinline__ void load(MsSmem &s) const
    {
        const uint32_t S = d->S;
        for (uint32_t i = threadIdx.x; i < S * 256u; i += blockDim.x) (&s.cum[0][0])[i] = (&d->cum[0][0])[i];
        for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) {
            s.C[i] = d->C[i];
            s.code_of_sym[i] = d->cum[S][i] ? i : 0xFFFFu;
        }
        for (uint32_t i = threadIdx.x; i <= S; i += blockDim.x) s.start[i] = d->start[i];
        if (threadIdx.x == 0) {
            // c0 = bwt[row0] = text[n-1] as a byte, fix = whether c0 occurs before row0; both 0 without a sampled SA
            const uint64_t row0 = d->row0;
            s.S = S;
            s.row0 = row0;
            s.c0 = 0;
            s.fix = 0;
            if (row0 < d->n) {
                const MsStep t = step(d->start, ms_slice_of(d->start, S, row0), row0);
                s.c0 = t.sym;
                s.fix = (d->cum[t.slice][t.sym] + t.occ) != 0;
            }
        }
    }
    // both boundaries of a backward-search step: a <- occ(ch, a), b <- occ(ch, b)
    __device__ __forceinline__ void rank2(const MsSmem &s, uint32_t, uint32_t ch, uint64_t &a, uint64_t &b) const
    {
        a = rank(s, ch, a);
        b = rank(s, ch, b);
    }
    __device__ __forceinline__ uint64_t rank(const MsSmem &s, uint32_t ch, uint64_t i) const
    {
        const uint32_t sl = ms_slice_of(s.start, s.S, i);
        const WtDev &w = d->slice[sl];
        const uint32_t code = __ldg(&w.tab->code_of_sym[ch]);
        const uint32_t local = code == 0xFFFFu ? 0u : wt_rank_code(*w.tab, w, code, (uint32_t)(i - s.start[sl]));
        return s.cum[sl][ch] + local;
    }
    // bwt[j] and its occurrences before j in the slice: the access + rank descent of slice sl (the slice holding j
    // among `start`), for a caller that has looked the slice up already
    __device__ __forceinline__ MsStep step(const uint64_t *start, uint32_t sl, uint64_t j) const
    {
        MsStep t;
        t.slice = sl;
        const WtDev &w = d->slice[sl];
        const uint32_t code = wt_access_rank(*w.tab, w, (uint32_t)(j - start[sl]), t.occ);
        t.sym = __ldg(&w.tab->sym_of_code[code]);
        return t;
    }
    __device__ __forceinline__ MsStep step(const MsSmem &s, uint64_t j) const
    {
        return step(s.start, ms_slice_of(s.start, s.S, j), j);
    }
    // the exact LF step: the global occ goes into lf_fix, so that row0 lands on C[c0]
    __device__ __forceinline__ uint64_t next(const MsSmem &s, const MsStep &t, uint64_t j) const
    {
        return s.C[t.sym] + lf_fix(s.cum[t.slice][t.sym] + t.occ, t.sym, j, s.c0, s.row0, s.fix);
    }
};

}  // namespace hkcsa
