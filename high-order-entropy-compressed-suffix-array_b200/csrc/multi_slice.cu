// multi_slice.cu -- the descriptor of the sliced index of the distributed build (BASELINE config 5): slice s covers
// global rows [start[s], start[s+1]) and carries its own wavelet tree (built over its BWT slice with libhkcsa K3) and
// its own sampled-SA marks/samples.  occ(c, i) over the whole BWT = (occurrences of c in the slices before the one
// holding i) + a rank walk inside that slice, so the recurrences of EnhancedFMIndex.find_range (reference
// csa/enhanced_fm_index.py:21-32) run unchanged on global row numbers.  Every GPU holds all slices (they are
// all-gathered after the build); patterns are sharded as in config 4.  The descriptor and its rank source MsDev are in
// multi_slice.cuh; count and locate over it are in fm_search.cu, extract in extract.cu.
#include "common.cuh"
#include "multi_slice.cuh"

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
