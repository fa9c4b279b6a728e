// dist_sa.cu -- distributed suffix-array construction (BASELINE config 5: a text beyond one GPU's working set;
// the reference's build_suffix_array, csa/suffix_array.py:131-134, sorts any text -- so does this).
//
// One process per GPU, `world` ranks.  The text is replicated (one all-gather; it is needed by the BWT gather
// anyway); everything else is partitioned:
//
//   1. every rank keys the suffixes of ITS block of positions with the same order-preserving prefix code as the
//      single-GPU builder (first bits0 bits of the code stream) and histograms the top 16 key bits; the
//      histograms are all-gathered and every rank derives the same balanced cut points: rank r owns the suffixes
//      whose bucket lies in [cuts[r], cuts[r+1]);
//   2. ONE kernel packs the keys of the block again, partitions each tile by destination in shared memory and
//      stores the (key, suffix id) runs straight into the owners' receive arrays through peer-mapped pointers
//      (NVLink) -- the all-to-all bucket exchange is part of the pack kernel, no collective follows it;
//   3. every rank radix-sorts what it received (onesweep) and refines its groups: first by EXTENSION rounds that
//      read the next symbols from the replicated text (no communication), then -- for whatever survives, i.e.
//      repetitive texts -- by RANK DOUBLING: the rank of suffix i + h is read from the position owner's ISA block
//      through its peer-mapped pointer (suffixes that were already unique before the switch never got an entry: their
//      rank is found by a binary search in the owner's sorted slice, comparing text), new ranks are stored
//      straight into the owners' ISA blocks; ranks synchronise between the read and the write phase of a round.
//
// The slices concatenated in rank order are the suffix array.  Suffix ids are 32-bit up to n = 2^32-2, 64-bit
// beyond (the sort then moves 32-bit ordinals, the ids stay in the receive array).
#include "common.cuh"
#include "prof.cuh"
#include "radix_sort.cuh"
#include "suffix_array.cuh"
#include <type_traits>

namespace hkcsa {

constexpr int DSA_BUCKET_BITS = 16;
constexpr int DSA_MAX_WORLD = HKCSA_DSA_MAX_RANKS;
// 64-bit suffix ids (n <= 2^40) travel with the BWT symbol of their suffix in the top byte: the source rank has
// text[i - 1] at hand when it packs suffix i, so the owner's BWT slice needs no random gather over the whole text
constexpr uint64_t DSA_ID_MASK = WIDE_ID_MASK;     // suffix_array.cuh: id in the low 40 bits, key extension above, BWT symbol on top

struct DsaDest {                       // kernel parameter of the exchange
    uint64_t *keys[DSA_MAX_WORLD];     // receive arrays of every rank (peer-mapped)
    void *ids[DSA_MAX_WORLD];          // uint32 ids, uint64 when WIDE
    uint64_t base[DSA_MAX_WORLD];      // first slot of THIS source's region in every destination
    uint32_t cuts[DSA_MAX_WORLD + 1];  // bucket boundaries
    uint32_t world;
};

__device__ __forceinline__ uint32_t dsa_dest_of(const uint32_t *cuts, uint32_t world, uint32_t bucket)
{
    uint32_t d = 0;
    for (uint32_t r = 1; r < world; ++r) d += (bucket >= cuts[r]) ? 1u : 0u;
    return d;
}

// MODE 0: histogram of the buckets (top 16 key bits) of suffixes [begin, end) -- of every tile_stride-th tile.
// MODE 1: (key, id) of every suffix of [begin, end) stored into the receive arrays of the rank owning its bucket.
// MODE 2: suffixes of [begin, end) per destination rank (counters[d]): the exact region sizes of the exchange when
//         the cut points came from a sampled histogram.
// Keys come from the same key source as the single-GPU builder's (AlphaKeys), so every mode and both builders agree on
// every key.
template <int MODE, bool WIDE>
__global__ void __launch_bounds__(PACK_THREADS, 4)
dsa_pack_kernel(const uint8_t *__restrict__ text, uint64_t n, uint64_t begin, uint64_t end, AlphaKeys src, int bits,
                DsaDest dd, unsigned long long *__restrict__ counters, unsigned long long *__restrict__ bucket_hist,
                uint32_t tile_stride, int xbits = 0)
{
    using IdT = typename std::conditional<WIDE, uint64_t, uint32_t>::type;
    __shared__ AlphaKeys::Smem s;
    __shared__ uint32_t s_cnt[DSA_MAX_WORLD], s_first[DSA_MAX_WORLD + 1], s_cuts[DSA_MAX_WORLD + 1];
    __shared__ uint64_t s_gbase[DSA_MAX_WORLD];
    __shared__ uint64_t *s_kptr[DSA_MAX_WORLD];
    __shared__ IdT *s_iptr[DSA_MAX_WORLD];
    __shared__ __align__(16) uint64_t s_keys[MODE == 1 ? PACK_TILE : 1];
    __shared__ __align__(16) IdT s_ids[MODE == 1 ? PACK_TILE : 1];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    src.setup(s);
    if (tid < DSA_MAX_WORLD) {
        s_cnt[tid] = 0;
        s_kptr[tid] = dd.keys[tid];
        s_iptr[tid] = static_cast<IdT *>(dd.ids[tid]);
    }
    if (tid <= DSA_MAX_WORLD) s_cuts[tid] = dd.cuts[tid];
    __syncthreads();
    const uint64_t base = begin + (uint64_t)blockIdx.x * tile_stride * PACK_TILE;
    const bool aligned8 = (reinterpret_cast<uintptr_t>(text + base) & 7) == 0;
    src.fill(s, text, n, base, aligned8);
    uint64_t key[PACK_IPT];
    uint32_t ds[PACK_IPT];            // MODE 1: destination << 16 | slot among the tile's elements for that destination
    uint16_t xk[MODE == 1 && WIDE ? PACK_IPT : 1];      // the WIDE_X_BITS code-stream bits that follow the key
    const uint32_t lt = lanemask_lt();
#pragma unroll
    for (int e = 0; e < PACK_IPT; ++e) {
        const uint32_t j = warp * (32u * PACK_IPT) + e * 32u + lane;
        const uint64_t g = base + j;
        // 64-bit ids leave room: the next 16 bits of the same code stream travel in the id word, so the group round
        // tells most tied suffixes apart without touching the text (xbits = 0: the look-ahead of the stream does not
        // reach that far for 1-bit code words -- the field stays zero, everything ties)
        uint16_t x = 0;
        key[e] = src.window(s, j, bits, MODE == 1 && WIDE ? &x : nullptr) >> (64 - bits);
        if (MODE == 1 && WIDE) xk[e] = xbits ? x : (uint16_t)0;
        const bool valid = g < end;
        const uint32_t bucket = (uint32_t)(key[e] >> (bits - DSA_BUCKET_BITS));
        if (MODE == 0) {
            const uint32_t b0 = __shfl_sync(0xffffffffu, bucket, 0);
            const uint32_t nv = __popc(__ballot_sync(0xffffffffu, valid));
            if (__all_sync(0xffffffffu, !valid || bucket == b0)) {      // runs of one symbol: one atomic per warp
                if (lane == 0 && nv) atomicAdd(&bucket_hist[b0], (unsigned long long)nv);
            } else if (valid) {
                atomicAdd(&bucket_hist[bucket], 1ull);
            }
        } else {
            const uint32_t dest = valid ? dsa_dest_of(s_cuts, dd.world, bucket) : 31u;
            const uint32_t peers = __match_any_sync(0xffffffffu, dest);
            const uint32_t leader = __ffs(peers) - 1;
            uint32_t first = 0;
            if (valid && lane == leader) first = atomicAdd(&s_cnt[dest], (uint32_t)__popc(peers));
            first = __shfl_sync(0xffffffffu, first, leader);
            ds[e] = (dest << 16) | (first + __popc(peers & lt));
        }
    }
    if (MODE == 0) return;
    __syncthreads();
    if (MODE == 2) {
        if (tid < dd.world && s_cnt[tid]) atomicAdd(&counters[tid], (unsigned long long)s_cnt[tid]);
        return;
    }
    if (tid < dd.world) {
        uint32_t pre = 0;
        for (uint32_t d = 0; d < tid; ++d) pre += s_cnt[d];
        s_first[tid] = pre;
        if (tid == dd.world - 1) s_first[dd.world] = pre + s_cnt[tid];
        // this source's region in destination `tid` starts at dd.base[tid]; tiles take their runs in arrival order
        s_gbase[tid] = dd.base[tid] + (s_cnt[tid] ? atomicAdd(&counters[tid], (unsigned long long)s_cnt[tid]) : 0ull);
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < PACK_IPT; ++e) {
        const uint32_t dest = ds[e] >> 16;
        if (dest != 31u) {
            const uint32_t j = warp * (32u * PACK_IPT) + e * 32u + lane;
            const uint32_t slot = s_first[dest] + (ds[e] & 0xFFFFu);
            s_keys[slot] = key[e];
            const uint64_t g = base + j;
            if (WIDE) s_ids[slot] = (IdT)(g | ((uint64_t)xk[e] << WIDE_ID_BITS) | ((uint64_t)text[g ? g - 1 : n - 1] << 56));
            else s_ids[slot] = (IdT)g;
        }
    }
    __syncthreads();
    // coalesced runs, one per destination, straight into the owners' arrays
    const uint32_t total = s_first[dd.world];
    for (uint32_t i = tid; i < total; i += PACK_THREADS) {
        uint32_t d = 0;
        while (i >= s_first[d + 1]) ++d;
        const uint64_t at = s_gbase[d] + (i - s_first[d]);
        s_kptr[d][at] = s_keys[i];
        s_iptr[d][at] = s_ids[i];
    }
}

// key of suffix g at depth `skip`: the next `k` symbol codes (b bits each), MSB first; 0 past the end
__device__ __forceinline__ uint64_t pack_from_text(const uint8_t *__restrict__ text, uint64_t n, uint64_t g,
                                                   const uint16_t *s_code, int b, int k)
{
    uint64_t key = 0;
    for (int q = 0; q < k; ++q) {
        const uint64_t t = g + q;
        key = (key << b) | (t < n ? (uint64_t)s_code[text[t]] : 0ull);
    }
    return key;
}

// extension round: key[j] = (group start << eb) | next `ke` symbols of suffix cidx[j] at depth `depth`
__global__ void __launch_bounds__(256)
dsa_keybuild_ext_kernel(const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp,
                        const uint8_t *__restrict__ text, uint64_t n, uint64_t depth, int b, int ke, int eb,
                        uint32_t m, int passes, CodeMap map, uint64_t *__restrict__ keys, uint32_t *__restrict__ ghist,
                        const uint64_t *__restrict__ ids64)
{
    __shared__ uint32_t s_hist[8 * RADIX];
    __shared__ uint16_t s_code[256];
    s_code[threadIdx.x] = map.code[threadIdx.x];
    hist_zero(s_hist, passes);
    __syncthreads();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < m; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t j = base + threadIdx.x;
        const bool valid = j < m;
        uint64_t key = 0;
        if (valid) {
            const uint64_t g = (ids64 ? (ids64[cidx[j]] & DSA_ID_MASK) : (uint64_t)cidx[j]) + depth;
            key = ((uint64_t)cgrp[j] << eb) | pack_from_text(text, n, g, s_code, b, ke);
            keys[j] = key;
        }
        hist_add_key(s_hist, key, passes, valid);
    }
    __syncthreads();
    hist_flush(s_hist, ghist, passes);
}

// ---------------------------------------------------------------- rank doubling over peer memory
struct DsaPeers {                          // kernel parameter of the doubling kernels
    void *isa[DSA_MAX_WORLD];              // ISA block of every rank: global rank of suffix blk * r + i at [i]
    const uint32_t *sa[DSA_MAX_WORLD];     // sorted slice of every rank (ids, or ordinals into ids64 when WIDE)
    const uint64_t *ids64[DSA_MAX_WORLD];  // WIDE: the received 64-bit ids of every rank
    uint64_t slice_off[DSA_MAX_WORLD + 1]; // global SA position of every slice's first entry
    uint32_t cuts[DSA_MAX_WORLD + 1];
    uint64_t blk;                          // positions per ISA block
    uint32_t world;
};

template <typename T>
__device__ __forceinline__ T ld_sys(const T *p)
{
    return *reinterpret_cast<const volatile T *>(p);        // peer memory: never from a stale L1 line
}

// order of two different suffixes by their symbols (the end of the text is smallest)
__device__ __forceinline__ bool suffix_less(const uint8_t *__restrict__ text, uint64_t n, uint64_t a, uint64_t b)
{
    while (true) {
        if (a >= n) return true;           // a is a proper prefix of b
        if (b >= n) return false;
        const uint32_t ca = text[a], cb = text[b];
        if (ca != cb) return ca < cb;
        ++a;
        ++b;
    }
}

// final rank of suffix t, which was already unique when rank doubling started (no ISA entry was ever written for
// it): binary search in the sorted slice of the rank owning its bucket.  Slots of groups still being refined hold
// SOME member of the group; t differs from all of them within the depth at which it became unique, so every
// comparison is decided by the symbols before that depth whatever member sits in the slot.
template <bool WIDE>
__device__ uint64_t dsa_remote_rank(const DsaPeers &pp, const uint8_t *__restrict__ text, uint64_t n, uint64_t t,
                                    const AlphaKeys::Tab &s_tab)
{
    const uint32_t bucket = (uint32_t)AlphaKeys::at(s_tab, text, n, t, DSA_BUCKET_BITS);
    const uint32_t r = dsa_dest_of(pp.cuts, pp.world, bucket);
    const uint32_t *sa = pp.sa[r];
    uint64_t lo = 0, hi = pp.slice_off[r + 1] - pp.slice_off[r];
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        uint64_t s = ld_sys(sa + mid);
        if (WIDE) s = ld_sys(pp.ids64[r] + s) & DSA_ID_MASK;
        if (s == t) return pp.slice_off[r] + mid;
        if (suffix_less(text, n, s, t)) lo = mid + 1; else hi = mid;
    }
    return pp.slice_off[r] + lo;
}

// key[j] = (group start << b2) | (global rank of suffix id + h, plus 1; 0 past the end)
template <typename IsaT, bool WIDE>
__global__ void __launch_bounds__(256)
dsa_keybuild_dbl_kernel(const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp, uint32_t m,
                        const uint8_t *__restrict__ text, uint64_t n, uint64_t h, int b2, int passes, AlphaCode ac,
                        DsaPeers pp, const uint64_t *__restrict__ ids64, uint64_t *__restrict__ keys,
                        uint32_t *__restrict__ ghist)
{
    __shared__ uint32_t s_hist[8 * RADIX];
    __shared__ AlphaKeys::Tab s_tab;
    s_tab.load(ac);
    hist_zero(s_hist, passes);
    __syncthreads();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < m; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t j = base + threadIdx.x;
        const bool valid = j < m;
        uint64_t key = 0;
        if (valid) {
            const uint64_t id = WIDE ? (ids64[cidx[j]] & DSA_ID_MASK) : (uint64_t)cidx[j];
            const uint64_t t = id + h;
            uint64_t k2 = 0;
            if (t < n) {
                const uint64_t owner = t / pp.blk;
                const IsaT v = ld_sys(static_cast<const IsaT *>(pp.isa[owner]) + (t - owner * pp.blk));
                k2 = (v == (IsaT)~(IsaT)0 ? dsa_remote_rank<WIDE>(pp, text, n, t, s_tab) : (uint64_t)v) + 1ull;
            }
            key = ((uint64_t)cgrp[j] << b2) | k2;
            keys[j] = key;
        }
        hist_add_key(s_hist, key, passes, valid);
    }
    __syncthreads();
    hist_flush(s_hist, ghist, passes);
}

// ISA[id] = slice_off + group start for the m_keep survivors (cidx, cgrp) of the last refinement and -- when
// m_sorted > 0 -- ISA[id] = slice_off + own slot for the elements of that round that became singletons (their
// final rank), so that later rounds read them from the ISA instead of searching.
template <typename IsaT, bool WIDE>
__global__ void __launch_bounds__(256)
dsa_isa_publish_kernel(const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cgrp, uint32_t m_keep,
                       const uint16_t *__restrict__ flags, const uint32_t *__restrict__ sidx,
                       const uint32_t *__restrict__ pos, uint32_t m_sorted, const uint64_t *__restrict__ ids64,
                       DsaPeers pp, uint64_t slice_off)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t j = t0; j < m_keep; j += stride) {
        const uint64_t id = WIDE ? (ids64[cidx[j]] & DSA_ID_MASK) : (uint64_t)cidx[j];
        const uint64_t owner = id / pp.blk;
        static_cast<IsaT *>(pp.isa[owner])[id - owner * pp.blk] = (IsaT)(slice_off + cgrp[j]);
    }
    for (uint64_t j = t0; j < m_sorted; j += stride) {
        const uint32_t f = flags[j >> 3];                     // bit e: head, bit 8 + e: singleton (seg_reduce_kernel)
        if ((f >> (SEG_IPT + (j & 7u))) & 1u) {
            const uint64_t id = WIDE ? (ids64[sidx[j]] & DSA_ID_MASK) : (uint64_t)sidx[j];
            const uint64_t owner = id / pp.blk;
            static_cast<IsaT *>(pp.isa[owner])[id - owner * pp.blk] = (IsaT)(slice_off + (pos ? pos[j] : (uint32_t)j));
        }
    }
}

template <typename IdT>
__global__ void bwt_slice_kernel(const uint8_t *__restrict__ text, uint64_t n, const IdT *__restrict__ sa,
                                 uint64_t m, uint8_t *__restrict__ out)
{
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint64_t v = sa[j];
    out[j] = text[v ? v - 1 : n - 1];
}

// the finished slice with 64-bit ids: id and BWT symbol of the j-th suffix from ONE random read
// Four consecutive rows per thread: one 16-byte load of ordinals, four independent random 8-byte reads in flight
// (the gather is bound by the rate of random requests), 2 x 16 bytes of ids and 4 BWT bytes stored.
__global__ void __launch_bounds__(256)
gather_ids64_kernel(const uint64_t *__restrict__ ids64, const uint32_t *__restrict__ ord, uint64_t m,
                    uint64_t *__restrict__ out, uint8_t *__restrict__ out_bwt)
{
    const uint64_t j0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (j0 >= m) return;
    const bool full = j0 + 4 <= m && ((reinterpret_cast<uintptr_t>(ord) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    uint32_t o[4] = {0, 0, 0, 0};
    if (full) {
        const uint4 q = __ldcs(reinterpret_cast<const uint4 *>(ord + j0));
        o[0] = q.x; o[1] = q.y; o[2] = q.z; o[3] = q.w;
    } else {
        for (int e = 0; e < 4; ++e) if (j0 + e < m) o[e] = ord[j0 + e];
    }
    uint64_t v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = (j0 + e < m) ? __ldg(ids64 + o[e]) : 0ull;
    if (full) {
        __stcs(reinterpret_cast<ulonglong2 *>(out + j0), make_ulonglong2(v[0] & DSA_ID_MASK, v[1] & DSA_ID_MASK));
        __stcs(reinterpret_cast<ulonglong2 *>(out + j0 + 2), make_ulonglong2(v[2] & DSA_ID_MASK, v[3] & DSA_ID_MASK));
        if (out_bwt) {
            const uint32_t w = (uint32_t)(v[0] >> 56) | ((uint32_t)(v[1] >> 56) << 8) | ((uint32_t)(v[2] >> 56) << 16) |
                               ((uint32_t)(v[3] >> 56) << 24);
            if ((reinterpret_cast<uintptr_t>(out_bwt) & 3) == 0) *reinterpret_cast<uint32_t *>(out_bwt + j0) = w;
            else for (int e = 0; e < 4; ++e) out_bwt[j0 + e] = (uint8_t)(w >> (8 * e));
        }
    } else {
        for (int e = 0; e < 4 && j0 + e < m; ++e) {
            out[j0 + e] = v[e] & DSA_ID_MASK;
            if (out_bwt) out_bwt[j0 + e] = (uint8_t)(v[e] >> 56);
        }
    }
}

// ---------------------------------------------------------------- host state of one rank's slice
struct DsaState {
    uint64_t magic;
    uint64_t n, M, m, depth, m_sorted;
    uint32_t round, wide, rounds_ext, rounds_dbl;
    int b, ke, eb, gb, b2, pcur;
    const uint8_t *text;
    const uint64_t *ids64;
    uint64_t *skey, *kx, *ky;
    uint32_t *sa, *sidx, *vfree, *vother;
    const uint32_t *pos;          // slots of the elements of the last sorted round (nullptr = identity: round 0)
    uint32_t *posbuf[2], *grp, *agg_head, *agg_keep, *counter, *cpos, *cidx;
    uint16_t *flags;
    SortScratch sort;
    uint64_t round_elems[48];
    CodeMap map;
    AlphaCode ac;
};
constexpr uint64_t DSA_MAGIC = 0x31415344414B4853ull;
static_assert(sizeof(DsaState) <= sizeof(hkcsa_dsa_state), "hkcsa_dsa_state too small");

struct DsaScratch {
    uint64_t *key;
    uint32_t *val;
    uint32_t *pos[2];
    uint32_t *grp, *agg_head, *agg_keep, *counter;
    uint16_t *flags;
    SortScratch sort;
};
static DsaScratch carve_dsa(Carver &c, uint64_t cap)
{
    DsaScratch b;
    const uint64_t tiles = (cap + SEG_TILE - 1) / SEG_TILE + 1;
    b.key = c.take<uint64_t>(cap);
    b.val = c.take<uint32_t>(cap);
    b.pos[0] = c.take<uint32_t>(cap);
    b.pos[1] = c.take<uint32_t>(cap);
    b.grp = c.take<uint32_t>(cap);
    b.agg_head = c.take<uint32_t>(tiles);
    b.agg_keep = c.take<uint32_t>(tiles);
    b.flags = c.take<uint16_t>(tiles * SEG_THREADS);
    b.counter = c.take<uint32_t>(64);
    b.sort = carve_sort_scratch(c, cap);
    return b;
}

// seg_reduce / seg_scan / seg_apply over the m sorted elements (S.skey, S.sidx, S.pos); reads the survivor count
static int dsa_refine(DsaState &S, cudaStream_t st)
{
    uint32_t *h_m = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(pinned_page()) + 2048);
    const uint32_t m = (uint32_t)S.m;
    const uint32_t tiles = (m + SEG_TILE - 1) / SEG_TILE;
    {
        prof::Scope ps(st, prof::SEG_REDUCE, (uint64_t)m * 8);
        seg_reduce_kernel<<<tiles, SEG_THREADS, 0, st>>>(S.skey, m, S.agg_head, S.agg_keep, S.flags, ~0ULL, nullptr);
        HK_LAUNCH_CHECK();
    }
    {
        prof::Scope ps(st, prof::SEG_SCAN, (uint64_t)tiles * 16);
        seg_scan_kernel<<<1, 1024, 0, st>>>(S.agg_head, S.agg_keep, tiles, S.counter);
        HK_LAUNCH_CHECK();
    }
    S.cpos = S.posbuf[S.pcur ^ 1];
    S.cidx = S.vfree;
    {
        prof::Scope ps(st, prof::SEG_APPLY, (uint64_t)m * 12);
        if (S.round == 0)      // nothing placed yet: the survivors only
            seg_compact0(S.flags, S.sidx, m, S.agg_head, S.agg_keep, S.cpos, S.cidx, S.grp, st);
        else
            seg_apply_kernel<<<tiles, SEG_THREADS, 0, st>>>(S.flags, S.sidx, S.pos, m, S.agg_head, S.agg_keep, S.sa,
                                                           nullptr, S.cpos, S.cidx, S.grp, true, false, nullptr, 0, nullptr);
        HK_LAUNCH_CHECK();
    }
    HK_CUDA(cudaMemcpyAsync(h_m, S.counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    S.m_sorted = m;
    if (S.round < 48) S.round_elems[S.round] = m;
    ++S.round;
    S.m = *h_m;
    return HKCSA_OK;
}

// sorts the keys built into S.kx for the current working set (values S.cidx) and refines
static int dsa_sort_refine(DsaState &S, int passes, cudaStream_t st)
{
    const uint32_t m = (uint32_t)S.m;
    if (S.round > 1) S.vother = S.sidx;                 // the sorted ids consumed by the last refinement: free again
    S.pcur ^= 1;
    S.pos = S.posbuf[S.pcur];
    uint32_t *vx = S.cidx, *vy = S.vother;
    HK_CUDA(radix_sort_pairs_u64(S.kx, vx, S.ky, vy, m, passes, S.sort, st));
    if (passes & 1) { S.skey = S.ky; S.sidx = vy; S.vfree = vx; uint64_t *t = S.kx; S.kx = S.ky; S.ky = t; }
    else { S.skey = S.kx; S.sidx = vx; S.vfree = vy; }
    if (S.skey == S.kx) { uint64_t *t = S.kx; S.kx = S.ky; S.ky = t; }   // kx never holds the sorted keys
    return dsa_refine(S, st);
}

static DsaState *dsa_state(hkcsa_dsa_state *p)
{
    DsaState *S = reinterpret_cast<DsaState *>(p);
    return (S && S->magic == DSA_MAGIC) ? S : nullptr;
}

static void fill_peers(DsaPeers &pp, const DsaState &S, uint32_t world, const uint64_t *h_peer_isa,
                       const uint64_t *h_peer_sa, const uint64_t *h_peer_ids64, const uint64_t *h_slice_off,
                       const uint32_t *h_cuts, uint64_t blk)
{
    memset(&pp, 0, sizeof(pp));
    for (uint32_t r = 0; r < world; ++r) {
        pp.isa[r] = reinterpret_cast<void *>(h_peer_isa[r]);
        if (h_peer_sa) pp.sa[r] = reinterpret_cast<const uint32_t *>(h_peer_sa[r]);
        if (h_peer_ids64) pp.ids64[r] = reinterpret_cast<const uint64_t *>(h_peer_ids64[r]);
    }
    if (h_slice_off) for (uint32_t r = 0; r <= world; ++r) pp.slice_off[r] = h_slice_off[r];
    if (h_cuts) for (uint32_t r = 0; r <= world; ++r) pp.cuts[r] = h_cuts[r];
    pp.blk = blk;
    pp.world = world;
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" size_t hkcsa_dsa_state_bytes(void) { return sizeof(hkcsa_dsa_state); }

extern "C" int hkcsa_dsa_plan_make(const uint64_t *h_byte_hist, uint64_t n, int force_wide, hkcsa_dsa_plan *p)
{
    HK_REQUIRE(h_byte_hist && p, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n <= (1ull << 40), HKCSA_ERANGE, "n exceeds 2^40");
    memset(p, 0, sizeof(*p));
    static thread_local Round0Plan r0;
    if (int rc = plan_round0(h_byte_hist, r0)) return rc;
    p->n = n;
    p->sigma = r0.sigma;
    p->bits0 = (uint32_t)r0.bits0;
    p->k0 = (uint32_t)r0.k0;
    p->passes0 = (uint32_t)r0.passes0;
    p->b_fixed = (uint32_t)r0.b;
    p->wide = (force_wide || n > HKCSA_DSA_MAX_N32) ? 1u : 0u;
    memcpy(p->code, r0.ac.code, sizeof(p->code));
    memcpy(p->len, r0.ac.len, sizeof(p->len));
    uint16_t code = 0;
    for (int ch = 0; ch < 256; ++ch) p->fixed_code[ch] = h_byte_hist[ch] ? ++code : (uint16_t)0;
    return HKCSA_OK;
}

static void plan_codes(const hkcsa_dsa_plan *p, AlphaCode &ac, CodeMap *map)
{
    memcpy(ac.code, p->code, sizeof(ac.code));
    memcpy(ac.len, p->len, sizeof(ac.len));
    if (map) memcpy(map->code, p->fixed_code, sizeof(map->code));
}

// the round-0 key source of plan p.  max_len = PACK_MAX_LEN: a tile clears its whole stream, because the key
// extension bits read the stream words behind the last code word.
static void plan_keys(const hkcsa_dsa_plan *p, AlphaKeys &src)
{
    plan_codes(p, src.code, nullptr);
    src.max_len = PACK_MAX_LEN;
}

// tile_stride > 1: only every tile_stride-th tile of 2048 positions is counted (cut points from a sample; the exact
// region sizes then come from hkcsa_dsa_dest_counts)
extern "C" int hkcsa_dsa_bucket_hist_sampled(const uint8_t *d_text, const hkcsa_dsa_plan *p, uint64_t begin, uint64_t end,
                                             uint32_t tile_stride, uint64_t *d_hist, void *stream)
{
    HK_REQUIRE(d_text && p && d_hist && tile_stride >= 1, HKCSA_EINVAL, "bad argument");
    HK_REQUIRE(begin <= end && end <= p->n, HKCSA_ERANGE, "range");
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemsetAsync(d_hist, 0, (size_t)HKCSA_DSA_BUCKETS * sizeof(uint64_t), st));
    if (begin == end) return HKCSA_OK;
    static thread_local AlphaKeys src;
    plan_keys(p, src);
    DsaDest dd;
    memset(&dd, 0, sizeof(dd));
    const uint64_t tiles = (end - begin + PACK_TILE - 1) / PACK_TILE;
    const uint64_t blocks = (tiles + tile_stride - 1) / tile_stride;
    HK_REQUIRE(blocks <= 0x7FFFFFFFull, HKCSA_ERANGE, "block of positions too large for one launch");
    prof::Scope ps(st, prof::SA_PACK0, (end - begin) / tile_stride);
    dsa_pack_kernel<0, false><<<(uint32_t)blocks, PACK_THREADS, 0, st>>>(d_text, p->n, begin, end, src, (int)p->bits0, dd,
                                                                       nullptr,
                                                                       reinterpret_cast<unsigned long long *>(d_hist),
                                                                       tile_stride);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_dsa_bucket_hist(const uint8_t *d_text, const hkcsa_dsa_plan *p, uint64_t begin, uint64_t end,
                                     uint64_t *d_hist, void *stream)
{
    return hkcsa_dsa_bucket_hist_sampled(d_text, p, begin, end, 1, d_hist, stream);
}

// suffixes of [begin, end) per destination rank under the cut points h_cuts -> d_counts[HKCSA_DSA_MAX_RANKS]
extern "C" int hkcsa_dsa_dest_counts(const uint8_t *d_text, const hkcsa_dsa_plan *p, uint64_t begin, uint64_t end,
                                     uint32_t world, const uint32_t *h_cuts, uint64_t *d_counts, void *stream)
{
    HK_REQUIRE(d_text && p && h_cuts && d_counts, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(world >= 1 && world <= (uint32_t)DSA_MAX_WORLD, HKCSA_EINVAL, "1..HKCSA_DSA_MAX_RANKS ranks");
    HK_REQUIRE(begin <= end && end <= p->n, HKCSA_ERANGE, "range");
    HK_REQUIRE(h_cuts[0] == 0 && h_cuts[world] == HKCSA_DSA_BUCKETS, HKCSA_EINVAL, "cuts must span every bucket");
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemsetAsync(d_counts, 0, DSA_MAX_WORLD * sizeof(uint64_t), st));
    if (begin == end) return HKCSA_OK;
    static thread_local AlphaKeys src;
    plan_keys(p, src);
    DsaDest dd;
    memset(&dd, 0, sizeof(dd));
    for (uint32_t r = 0; r <= world; ++r) dd.cuts[r] = h_cuts[r];
    dd.world = world;
    const uint64_t blocks = (end - begin + PACK_TILE - 1) / PACK_TILE;
    HK_REQUIRE(blocks <= 0x7FFFFFFFull, HKCSA_ERANGE, "block of positions too large for one launch");
    prof::Scope ps(st, prof::SA_PACK0, end - begin);
    dsa_pack_kernel<2, false><<<(uint32_t)blocks, PACK_THREADS, 0, st>>>(d_text, p->n, begin, end, src, (int)p->bits0, dd,
                                                                       reinterpret_cast<unsigned long long *>(d_counts),
                                                                       nullptr, 1);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_dsa_pack_exchange(const uint8_t *d_text, const hkcsa_dsa_plan *p, uint64_t begin, uint64_t end,
                                       uint32_t world, const uint32_t *h_cuts, const uint64_t *h_peer_keys,
                                       const uint64_t *h_peer_ids, const uint64_t *h_base, uint64_t *d_counters,
                                       void *stream)
{
    HK_REQUIRE(d_text && p && h_cuts && h_peer_keys && h_peer_ids && h_base && d_counters, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(world >= 1 && world <= (uint32_t)DSA_MAX_WORLD, HKCSA_EINVAL, "1..HKCSA_DSA_MAX_RANKS ranks");
    HK_REQUIRE(begin <= end && end <= p->n, HKCSA_ERANGE, "range");
    HK_REQUIRE(h_cuts[0] == 0 && h_cuts[world] == HKCSA_DSA_BUCKETS, HKCSA_EINVAL, "cuts must span every bucket");
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemsetAsync(d_counters, 0, DSA_MAX_WORLD * sizeof(uint64_t), st));
    if (begin == end) return HKCSA_OK;
    static thread_local AlphaKeys src;
    plan_keys(p, src);
    DsaDest dd;
    memset(&dd, 0, sizeof(dd));
    for (uint32_t r = 0; r < world; ++r) {
        HK_REQUIRE(h_cuts[r] <= h_cuts[r + 1], HKCSA_EINVAL, "cuts must ascend");
        dd.keys[r] = reinterpret_cast<uint64_t *>(h_peer_keys[r]);
        dd.ids[r] = reinterpret_cast<void *>(h_peer_ids[r]);
        dd.base[r] = h_base[r];
    }
    for (uint32_t r = 0; r <= world; ++r) dd.cuts[r] = h_cuts[r];
    dd.world = world;
    const uint64_t blocks = (end - begin + PACK_TILE - 1) / PACK_TILE;
    HK_REQUIRE(blocks <= 0x7FFFFFFFull, HKCSA_ERANGE, "block of positions too large for one launch");
    // algorithmic bytes: 1 B of text read, 8 B key + 4 / 8 B id stored (over NVLink for remote owners)
    prof::Scope ps(st, prof::SA_PACK0, (end - begin) * (p->wide ? 17 : 13));
    unsigned long long *cnt = reinterpret_cast<unsigned long long *>(d_counters);
    // the stream of a tile reaches PACK_LOOK positions beyond it: 64 + WIDE_X_BITS bits exist for every position when
    // no code word is shorter than two bits
    int min_len = src.code.len[256];                            // past the end, then the bytes that occur
    for (int c = 0; c < 256; ++c) if (p->fixed_code[c] && src.code.len[c] < min_len) min_len = src.code.len[c];
    const int xbits = (min_len >= 2 && !getenv("HKCSA_DSA_NO_XBITS")) ? WIDE_X_BITS : 0;
    if (p->wide)
        dsa_pack_kernel<1, true><<<(uint32_t)blocks, PACK_THREADS, 0, st>>>(d_text, p->n, begin, end, src, (int)p->bits0, dd, cnt, nullptr, 1, xbits);
    else
        dsa_pack_kernel<1, false><<<(uint32_t)blocks, PACK_THREADS, 0, st>>>(d_text, p->n, begin, end, src, (int)p->bits0, dd, cnt, nullptr, 1);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" size_t hkcsa_dsa_scratch_bytes(uint64_t capacity)
{
    Carver c(nullptr);
    carve_dsa(c, capacity ? capacity : 1);
    return c.total();
}

extern "C" int hkcsa_dsa_begin(hkcsa_dsa_state *state, const hkcsa_dsa_plan *p, const uint8_t *d_text, uint64_t *d_keys,
                               void *d_ids, uint32_t *d_val_a, uint32_t *d_val_b, uint64_t M, uint64_t capacity,
                               void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(state && p && d_text && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(capacity <= HKCSA_MAX_N && M <= capacity, HKCSA_ERANGE, "slice exceeds HKCSA_MAX_N or its capacity");
    HK_REQUIRE(M == 0 || (d_keys && d_ids && d_val_a && d_val_b), HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(((reinterpret_cast<uintptr_t>(d_keys) | reinterpret_cast<uintptr_t>(d_val_a) |
                 reinterpret_cast<uintptr_t>(d_val_b) | reinterpret_cast<uintptr_t>(d_scratch)) & 15) == 0,
               HKCSA_EINVAL, "buffers must be 16-byte aligned (TMA bulk copies)");
    Carver c(d_scratch);
    DsaScratch B = carve_dsa(c, capacity ? capacity : 1);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "scratch too small");
    HK_REQUIRE(pinned_page() != nullptr, HKCSA_ECUDA, "pinned page allocation failed");
    cudaStream_t st = as_stream(stream);
    memset(state, 0, sizeof(*state));
    DsaState &S = *reinterpret_cast<DsaState *>(state);
    S.magic = DSA_MAGIC;
    S.n = p->n; S.M = M; S.m = M; S.wide = p->wide;
    S.text = d_text;
    S.ids64 = p->wide ? static_cast<const uint64_t *>(d_ids) : nullptr;
    plan_codes(p, S.ac, &S.map);
    S.b = std::max(1, (int)p->b_fixed);
    S.gb = (int)bits_for(capacity > 1 ? capacity - 1 : 1);   // bits of a group start; the same on every rank
    S.ke = std::max(1, (64 - S.gb) / S.b);                   // symbols per extension round
    S.eb = S.ke * S.b;
    S.b2 = (int)bits_for(p->n);                              // global rank + 1 <= n
    S.depth = p->k0;
    S.posbuf[0] = B.pos[0]; S.posbuf[1] = B.pos[1];
    S.grp = B.grp; S.agg_head = B.agg_head; S.agg_keep = B.agg_keep; S.counter = B.counter; S.flags = B.flags;
    S.sort = B.sort;
    S.pos = nullptr;
    S.pcur = 0;
    const int passes0 = (int)p->passes0;
    // narrow: d_val_a holds the received ids; wide: the values are ordinals 0, 1, ... into the received ids
    uint32_t *va = p->wide ? d_val_a : static_cast<uint32_t *>(d_ids);
    HK_REQUIRE(p->wide || static_cast<void *>(d_val_a) == d_ids, HKCSA_EINVAL, "narrow ids: d_val_a must be the id array");
    uint32_t *vb = d_val_b;
    S.sa = (passes0 % 2 == 0) ? va : vb;
    uint32_t *vrest = (passes0 % 2 == 0) ? vb : va;          // free after the round-0 sort
    uint64_t *ka = d_keys, *kb = B.key;
    if (M == 0) { S.m = 0; return HKCSA_OK; }
    HK_CUDA(radix_histogram_u64(ka, (uint32_t)M, passes0, S.sort, st));
    HK_CUDA(radix_sort_pairs_u64(ka, va, kb, vb, (uint32_t)M, passes0, S.sort, st, /*identity_vals=*/p->wide != 0));
    S.skey = (passes0 % 2 == 0) ? ka : kb;
    S.kx = (passes0 % 2 == 0) ? kb : ka;
    S.ky = S.skey;
    S.sidx = S.sa;
    S.vfree = B.val;
    S.vother = vrest;
    return dsa_refine(S, st);
}

extern "C" uint64_t hkcsa_dsa_working_set(const hkcsa_dsa_state *state)
{
    const DsaState *S = reinterpret_cast<const DsaState *>(state);
    return (S && S->magic == DSA_MAGIC) ? S->m : 0;
}
extern "C" uint64_t hkcsa_dsa_depth(const hkcsa_dsa_state *state)
{
    const DsaState *S = reinterpret_cast<const DsaState *>(state);
    return (S && S->magic == DSA_MAGIC) ? S->depth : 0;
}
extern "C" const void *hkcsa_dsa_slice(const hkcsa_dsa_state *state)
{
    const DsaState *S = reinterpret_cast<const DsaState *>(state);
    return (S && S->magic == DSA_MAGIC) ? S->sa : nullptr;
}
extern "C" int hkcsa_dsa_rounds(const hkcsa_dsa_state *state, uint32_t *h_rounds, uint64_t *h_round_elems, uint32_t max_rounds)
{
    const DsaState *S = reinterpret_cast<const DsaState *>(state);
    HK_REQUIRE(S && S->magic == DSA_MAGIC && h_rounds, HKCSA_EINVAL, "bad state");
    *h_rounds = S->round;
    for (uint32_t r = 0; h_round_elems && r < max_rounds && r < S->round && r < 48; ++r) h_round_elems[r] = S->round_elems[r];
    return HKCSA_OK;
}

// One extension round over the working set; every rank advances by the same number of symbols (ke follows from
// the common capacity), so the depth stays the same on all ranks.  A rank without survivors only advances its depth.
extern "C" int hkcsa_dsa_ext_round(hkcsa_dsa_state *state, void *stream)
{
    DsaState *Sp = dsa_state(state);
    HK_REQUIRE(Sp, HKCSA_EINVAL, "bad state");
    DsaState &S = *Sp;
    cudaStream_t st = as_stream(stream);
    if (S.m == 0) { S.depth += (uint64_t)S.ke; return HKCSA_OK; }
    const uint32_t m = (uint32_t)S.m;
    const int passes = (S.gb + S.eb + 7) / 8;
    HK_CUDA(cudaMemsetAsync(S.sort.hist, 0, 8 * RADIX * sizeof(uint32_t), st));
    {
        const int blocks = (int)std::min<uint64_t>(((uint64_t)m + 255) / 256, (uint64_t)num_sms() * 16);
        prof::Scope ps(st, prof::SA_KEYBUILD, (uint64_t)m * 20);
        dsa_keybuild_ext_kernel<<<blocks, 256, 0, st>>>(S.cidx, S.grp, S.text, S.n, S.depth, S.b, S.ke, S.eb, m, passes,
                                                        S.map, S.kx, S.sort.hist, S.ids64);
        HK_LAUNCH_CHECK();
    }
    S.depth += (uint64_t)S.ke;
    ++S.rounds_ext;
    return dsa_sort_refine(S, passes, st);
}

// One refinement round without a radix sort or communication: every group of at most GS_MAX suffixes is ordered by
// comparing the replicated text beyond the current depth (group_local_keys).  Meant for the first round after
// hkcsa_dsa_begin, when nearly all groups hold two or three suffixes.  The depth does not advance.
extern "C" int hkcsa_dsa_group_round(hkcsa_dsa_state *state, void *stream)
{
    DsaState *Sp = dsa_state(state);
    HK_REQUIRE(Sp, HKCSA_EINVAL, "bad state");
    DsaState &S = *Sp;
    if (S.m == 0) return HKCSA_OK;
    cudaStream_t st = as_stream(stream);
    const uint32_t m = (uint32_t)S.m;
    if (S.round > 1) S.vother = S.sidx;                 // the sorted ids consumed by the last refinement: free again
    S.pcur ^= 1;
    S.pos = S.posbuf[S.pcur];
    {
        prof::Scope ps(st, prof::SA_KEYBUILD, (uint64_t)m * 48);
        HK_CUDA(group_local_keys(S.cidx, S.grp, m, S.text, S.n, S.depth, false, S.ids64, S.kx, st));
    }
    S.skey = S.kx;
    S.sidx = S.cidx;
    S.vfree = S.vother;
    { uint64_t *t = S.kx; S.kx = S.ky; S.ky = t; }      // kx never holds the keys being refined
    return dsa_refine(S, st);
}

extern "C" int hkcsa_dsa_isa_publish(hkcsa_dsa_state *state, uint32_t world, const uint64_t *h_peer_isa, uint64_t blk,
                                     uint64_t slice_offset, int with_singles, void *stream)
{
    DsaState *Sp = dsa_state(state);
    HK_REQUIRE(Sp && h_peer_isa, HKCSA_EINVAL, "bad state or null pointer");
    HK_REQUIRE(world >= 1 && world <= (uint32_t)DSA_MAX_WORLD && blk >= 1, HKCSA_EINVAL, "bad world or block size");
    DsaState &S = *Sp;
    const uint32_t m_keep = (uint32_t)S.m;
    const uint32_t m_sorted = with_singles ? (uint32_t)S.m_sorted : 0u;
    if (m_keep == 0 && m_sorted == 0) return HKCSA_OK;
    cudaStream_t st = as_stream(stream);
    DsaPeers pp;
    fill_peers(pp, S, world, h_peer_isa, nullptr, nullptr, nullptr, nullptr, blk);
    const uint32_t work = std::max(m_keep, m_sorted);
    const int blocks = (int)std::min<uint64_t>(((uint64_t)work + 255) / 256, (uint64_t)num_sms() * 16);
    prof::Scope ps(st, prof::OTHER, (uint64_t)m_keep * 16 + (uint64_t)m_sorted * 2);
    if (S.wide)
        dsa_isa_publish_kernel<uint64_t, true><<<blocks, 256, 0, st>>>(S.cidx, S.grp, m_keep, S.flags, S.sidx, S.pos,
                                                                       m_sorted, S.ids64, pp, slice_offset);
    else
        dsa_isa_publish_kernel<uint32_t, false><<<blocks, 256, 0, st>>>(S.cidx, S.grp, m_keep, S.flags, S.sidx, S.pos,
                                                                        m_sorted, S.ids64, pp, slice_offset);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// Doubling round, read phase: keys (group start, rank of suffix id + depth) of the working set from the ISA blocks
// of all ranks.  The caller synchronises the ranks before hkcsa_dsa_dbl_sort (whose follow-up publish overwrites
// ISA entries that this phase reads on other ranks).
extern "C" int hkcsa_dsa_dbl_keys(hkcsa_dsa_state *state, uint32_t world, const uint64_t *h_peer_isa, uint64_t blk,
                                  const uint64_t *h_peer_sa, const uint64_t *h_peer_ids64, const uint64_t *h_slice_off,
                                  const uint32_t *h_cuts, void *stream)
{
    DsaState *Sp = dsa_state(state);
    HK_REQUIRE(Sp && h_peer_isa && h_peer_sa && h_slice_off && h_cuts, HKCSA_EINVAL, "bad state or null pointer");
    HK_REQUIRE(world >= 1 && world <= (uint32_t)DSA_MAX_WORLD && blk >= 1, HKCSA_EINVAL, "bad world or block size");
    DsaState &S = *Sp;
    HK_REQUIRE(!S.wide || h_peer_ids64, HKCSA_EINVAL, "64-bit ids need the id arrays of every rank");
    HK_REQUIRE(S.gb + S.b2 <= 64, HKCSA_ERANGE, "group start and global rank do not fit one 64-bit key");
    if (S.m == 0) return HKCSA_OK;
    cudaStream_t st = as_stream(stream);
    const uint32_t m = (uint32_t)S.m;
    const int passes = (S.gb + S.b2 + 7) / 8;
    DsaPeers pp;
    fill_peers(pp, S, world, h_peer_isa, h_peer_sa, h_peer_ids64, h_slice_off, h_cuts, blk);
    HK_CUDA(cudaMemsetAsync(S.sort.hist, 0, 8 * RADIX * sizeof(uint32_t), st));
    const int blocks = (int)std::min<uint64_t>(((uint64_t)m + 255) / 256, (uint64_t)num_sms() * 16);
    prof::Scope ps(st, prof::SA_KEYBUILD, (uint64_t)m * 24);
    if (S.wide)
        dsa_keybuild_dbl_kernel<uint64_t, true><<<blocks, 256, 0, st>>>(S.cidx, S.grp, m, S.text, S.n, S.depth, S.b2, passes,
                                                                        S.ac, pp, S.ids64, S.kx, S.sort.hist);
    else
        dsa_keybuild_dbl_kernel<uint32_t, false><<<blocks, 256, 0, st>>>(S.cidx, S.grp, m, S.text, S.n, S.depth, S.b2, passes,
                                                                         S.ac, pp, S.ids64, S.kx, S.sort.hist);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// Doubling round, local phase: sort the keys of hkcsa_dsa_dbl_keys and refine.  The depth doubles on every rank.
extern "C" int hkcsa_dsa_dbl_sort(hkcsa_dsa_state *state, void *stream)
{
    DsaState *Sp = dsa_state(state);
    HK_REQUIRE(Sp, HKCSA_EINVAL, "bad state");
    DsaState &S = *Sp;
    const uint64_t h = S.depth;
    S.depth = h * 2;
    ++S.rounds_dbl;
    if (S.m == 0) { S.m_sorted = 0; return HKCSA_OK; }
    HK_REQUIRE(h < S.n, HKCSA_EINVAL, "internal: groups remain after depth >= n");
    return dsa_sort_refine(S, (S.gb + S.b2 + 7) / 8, as_stream(stream));
}

// 64-bit ids: out[j] = ids[ordinal[j]] for the finished slice
extern "C" int hkcsa_dsa_gather_ids64(const hkcsa_dsa_state *state, uint64_t *d_out, uint8_t *d_out_bwt, void *stream)
{
    const DsaState *S = reinterpret_cast<const DsaState *>(state);
    HK_REQUIRE(S && S->magic == DSA_MAGIC && S->wide, HKCSA_EINVAL, "bad state (64-bit ids only)");
    if (S->M == 0) return HKCSA_OK;
    HK_REQUIRE(d_out, HKCSA_EINVAL, "null pointer");
    prof::Scope ps(as_stream(stream), prof::BWT_GATHER, S->M * 21);
    gather_ids64_kernel<<<(uint32_t)((S->M + 1023) / 1024), 256, 0, as_stream(stream)>>>(S->ids64, S->sa, S->M, d_out, d_out_bwt);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_bwt_slice(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa_slice, uint64_t m,
                               uint8_t *d_out, void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_text && d_sa_slice && d_out, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n <= HKCSA_DSA_MAX_N32, HKCSA_ERANGE, "n exceeds 2^32-2");
    prof::Scope ps(as_stream(stream), prof::BWT_GATHER, m * 6);
    bwt_slice_kernel<uint32_t><<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(d_text, n, d_sa_slice, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_bwt_slice64(const uint8_t *d_text, uint64_t n, const uint64_t *d_sa_slice, uint64_t m,
                                 uint8_t *d_out, void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_REQUIRE(d_text && d_sa_slice && d_out, HKCSA_EINVAL, "null pointer");
    prof::Scope ps(as_stream(stream), prof::BWT_GATHER, m * 10);
    bwt_slice_kernel<uint64_t><<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(d_text, n, d_sa_slice, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
