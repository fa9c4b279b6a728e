// multi_slice.cuh -- the descriptor of the sliced index (multi_slice.cu), shared with the cross-slice extract walk
// (extract.cu).
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
__device__ __forceinline__ uint32_t ms_slice_of(const MultiDesc *d, uint64_t i) { return ms_slice_of(d->start, d->S, i); }

// What the exact LF step (lf_fix) needs, read once per CTA: c0 = bwt[row0] = text[n-1] as a byte, and fix = whether
// c0 occurs before row0.  Both 0 without a sampled SA.
__device__ __forceinline__ void ms_suffix0(const MultiDesc *d, uint32_t &c0, uint32_t &fix)
{
    c0 = 0;
    fix = 0;
    const uint64_t row0 = d->row0;
    if (row0 < d->n) {
        const uint32_t s = ms_slice_of(d, row0);
        const WtDev &w = d->slice[s];
        uint32_t occ0;
        const uint32_t code = wt_access_rank(*w.tab, w, (uint32_t)(row0 - d->start[s]), occ0);
        c0 = w.tab->sym_of_code[code];
        fix = (d->cum[s][c0] + occ0) != 0;
    }
}

}  // namespace hkcsa
