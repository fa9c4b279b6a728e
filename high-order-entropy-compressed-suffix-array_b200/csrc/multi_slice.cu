// multi_slice.cu -- FM backward search over a BWT that was built in slices (distributed build, BASELINE
// config 5): slice s covers global rows [start[s], start[s+1]) and carries its own wavelet tree (built over its
// BWT slice with libhkcsa K3) and its own sampled-SA marks/samples.  occ(c, i) over the whole BWT =
// (occurrences of c in the slices before the one holding i) + a rank walk inside that slice, so the recurrences
// of EnhancedFMIndex.find_range (reference csa/enhanced_fm_index.py:21-32) run unchanged on global row numbers.
// Every GPU holds all slices (they are all-gathered after the build); patterns are sharded as in config 4.
// The descriptor (MultiDesc) is in multi_slice.cuh; extract.cu walks the same index across slices.
#include "common.cuh"
#include "multi_slice.cuh"
#include "prof.cuh"
#include "wavelet.cuh"

namespace hkcsa {

// occurrences of `byte` in global rows [0, i)
__device__ __forceinline__ uint64_t ms_rank(const MultiDesc *d, uint32_t byte, uint64_t i)
{
    const uint32_t s = ms_slice_of(d, i);
    const WtDev &w = d->slice[s];
    const uint32_t code = __ldg(&w.tab->code_of_sym[byte]);
    uint32_t local = 0;
    if (code != 0xFFFFu) {
        const uint32_t p = (uint32_t)(i - d->start[s]);
        local = (w.sigma == 1) ? p : wt_rank_code(*w.tab, w, code, p);   // node tables from global memory
    }
    return d->cum[s][byte] + local;
}

__global__ void __launch_bounds__(256)
ms_count_kernel(const MultiDesc *__restrict__ d, const uint8_t *__restrict__ pat, const int64_t *__restrict__ off,
                uint64_t P, int64_t *__restrict__ out_lo, int64_t *__restrict__ out_hi)
{
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int64_t b = off[p], e = off[p + 1];
    uint64_t l = 0, r = d->n;
    bool miss = false;
    for (int64_t k = e - 1; k >= b; --k) {
        const uint32_t c = pat[k];
        if (d->cum[d->S][c] == 0) { miss = true; break; }       // symbol absent from the text
        l = d->C[c] + ms_rank(d, c, l);
        r = d->C[c] + ms_rank(d, c, r);
        if (l >= r) { miss = true; break; }
    }
    out_lo[p] = miss ? -1 : (int64_t)l;
    out_hi[p] = miss ? -1 : (int64_t)r - 1;
}

// text position of global row j: LF walk across slices until a marked row.  The step is the exact one of
// locate_rows_kernel (lf_fix, csrc/common.cuh) on global rows and byte symbols: slices number their codes apart.
// Kept apart from locate_rows_kernel (fm_search.cu): one slice lookup per step serves both the mark test and the LF
// step, and rows, C[] and positions are 64-bit.
__global__ void __launch_bounds__(256)
ms_locate_kernel(const MultiDesc *__restrict__ d, const uint64_t *__restrict__ rows, uint64_t m,
                 uint64_t *__restrict__ out)
{
    __shared__ uint32_t s_c0, s_fix;
    const uint64_t row0 = d->row0;
    if (threadIdx.x == 0) ms_suffix0(d, s_c0, s_fix);
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    uint64_t j = rows[q];
    uint32_t steps = 0;
    while (true) {
        const uint32_t s = ms_slice_of(d, j);
        const uint32_t lj = (uint32_t)(j - d->start[s]);
        uint64_t slot;
        if (marked_slot(d->marks[s], lj, slot)) {
            out[q] = (uint64_t)d->samples[s][slot] * d->rate + steps;
            return;
        }
        // with the exact step a walk meets a marked row within rate-1 steps on every text; the bound only keeps a
        // walk over a corrupt index from spinning
        if (steps >= d->rate) { out[q] = HKCSA_NO_POSITION64; return; }
        const WtDev &w = d->slice[s];
        uint32_t occ;
        const uint32_t code = wt_access_rank(*w.tab, w, lj, occ);
        const uint32_t byte = w.tab->sym_of_code[code];
        j = d->C[byte] + lf_fix(d->cum[s][byte] + occ, byte, j, s_c0, row0, s_fix);
        ++steps;
    }
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" size_t hkcsa_multi_desc_bytes(void) { return sizeof(MultiDesc); }

// h_starts: uint64[S+1] global first row of every slice (h_starts[S] = n).  d_ssa_blobs / h_ssa_plans may be
// NULL (no locate); row0 = the global row of suffix 0 (< n), UINT64_MAX without them.  Builds the descriptor on the
// host and copies it into d_desc (hkcsa_multi_desc_bytes()).  syncs.
extern "C" int hkcsa_multi_desc_build(uint32_t S, const void *const *d_wt_blobs, const hkcsa_wt_plan *const *h_plans,
                                      const uint64_t *h_starts, const void *const *d_ssa_blobs,
                                      const hkcsa_ssa_plan *const *h_ssa_plans, uint64_t row0, void *d_desc,
                                      void *stream)
{
    HK_REQUIRE(S >= 1 && S <= HKCSA_MAX_SLICES, HKCSA_EINVAL, "1..HKCSA_MAX_SLICES slices");
    HK_REQUIRE(d_wt_blobs && h_plans && h_starts && d_desc, HKCSA_EINVAL, "null pointer");
    static thread_local MultiDesc D;
    memset(&D, 0, sizeof(D));
    D.S = S;
    D.n = h_starts[S];
    HK_REQUIRE(D.n <= (1ull << 40), HKCSA_ERANGE, "n exceeds 2^40");
    uint64_t tot[256];
    memset(tot, 0, sizeof(tot));
    for (uint32_t s = 0; s < S; ++s) {
        HK_REQUIRE(d_wt_blobs[s] && h_plans[s], HKCSA_EINVAL, "null slice");
        HK_REQUIRE(h_plans[s]->n == h_starts[s + 1] - h_starts[s], HKCSA_EINVAL, "slice length != plan length");
        D.slice[s] = make_wt_dev(d_wt_blobs[s], h_plans[s]);
        D.start[s] = h_starts[s];
        for (int c = 0; c < 256; ++c) D.cum[s][c] = tot[c];
        for (uint32_t k = 0; k < h_plans[s]->sigma; ++k) tot[h_plans[s]->sym_of_code[k]] += h_plans[s]->cnt[k];
        if (d_ssa_blobs && h_ssa_plans && d_ssa_blobs[s] && h_ssa_plans[s]) {
            const uint8_t *sb = static_cast<const uint8_t *>(d_ssa_blobs[s]);
            D.marks[s].blocks = reinterpret_cast<const RankBlock *>(sb + h_ssa_plans[s]->off_blocks);
            D.marks[s].super = reinterpret_cast<const uint64_t *>(sb + h_ssa_plans[s]->off_super);
            D.marks[s].len = h_ssa_plans[s]->n;
            D.samples[s] = reinterpret_cast<const uint32_t *>(sb + h_ssa_plans[s]->off_samples);
            D.rate = h_ssa_plans[s]->rate;
        }
    }
    D.start[S] = h_starts[S];
    uint64_t run = 0;
    for (int c = 0; c < 256; ++c) {
        D.cum[S][c] = tot[c];
        D.C[c] = run;
        run += tot[c];
    }
    HK_REQUIRE(run == D.n, HKCSA_EINVAL, "slice symbol counts do not add up to n");
    HK_REQUIRE(row0 < D.n || (row0 == UINT64_MAX && D.rate == 0), HKCSA_EINVAL,
               "row0 (the row of suffix 0) out of range");
    D.row0 = row0;
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemcpyAsync(d_desc, &D, sizeof(D), cudaMemcpyHostToDevice, st));
    HK_CUDA(cudaStreamSynchronize(st));
    return HKCSA_OK;
}

extern "C" int hkcsa_multi_count_batch(const void *d_desc, const uint8_t *d_pat, const int64_t *d_off, uint64_t P,
                                       int64_t *d_lo, int64_t *d_hi, void *stream)
{
    if (P == 0) return HKCSA_OK;
    HK_REQUIRE(d_desc && d_off && d_lo && d_hi, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    prof::Scope ps(st, prof::COUNT, 0);
    ms_count_kernel<<<(uint32_t)((P + 255) / 256), 256, 0, st>>>(static_cast<const MultiDesc *>(d_desc), d_pat, d_off, P,
                                                                d_lo, d_hi);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_multi_locate_rows(const void *d_desc, const uint64_t *d_rows, uint64_t m, uint64_t *d_out_pos,
                                       void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_desc && d_rows && d_out_pos, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    prof::Scope ps(st, prof::LOCATE, 0);
    ms_locate_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, st>>>(static_cast<const MultiDesc *>(d_desc), d_rows, m,
                                                                 d_out_pos);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
