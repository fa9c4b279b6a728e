// radix_sort.cu -- onesweep LSD radix sort kernels (see radix_sort.cuh).
#include "radix_sort.cuh"
#include "prof.cuh"
#include <stdlib.h>

namespace hkcsa {

// VAL_MODE: 0 = keys only, 1 = values loaded from vin, 2 = value = source index.
template <typename KeyT, int VAL_MODE, int THREADS, int IPT>
__global__ void __launch_bounds__(THREADS)
onesweep_kernel(const KeyT *__restrict__ kin, KeyT *__restrict__ kout, const uint32_t *__restrict__ vin,
                uint32_t *__restrict__ vout, uint32_t n, int shift, const uint8_t *__restrict__ lut,
                const uint32_t *__restrict__ digit_base, uint32_t *lookback, uint32_t *ticket)
{
    constexpr int TILE = THREADS * IPT;
    constexpr int WARPS = THREADS / 32;
    constexpr bool BYTE_KEYS = (sizeof(KeyT) == 1);
    static_assert(THREADS >= RADIX, "one thread per digit is required");
    static_assert(WARPS <= 32, "warp totals live in s_misc");

    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint32_t *s_whist = reinterpret_cast<uint32_t *>(smem_raw);   // [WARPS][RADIX]
    uint32_t *s_gbase = s_whist + WARPS * RADIX;                  // [RADIX]
    uint32_t *s_misc = s_gbase + RADIX;                           // [64]
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(s_misc + 64);    // [256]
    KeyT *s_keys = reinterpret_cast<KeyT *>(s_lut + 256);         // [TILE]
    uint32_t *s_vals = reinterpret_cast<uint32_t *>(s_lut + 256); // [TILE] (aliases s_keys)

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

    if (tid == 0) s_misc[0] = atomicAdd(ticket, 1u);
    for (int i = tid; i < WARPS * RADIX; i += THREADS) s_whist[i] = 0;
    if (BYTE_KEYS && tid < 256) s_lut[tid] = lut[tid];
    __syncthreads();

    const uint32_t tile = s_misc[0];
    const uint32_t tile_base = tile * (uint32_t)TILE;
    const uint32_t nvalid = min((uint32_t)TILE, n - tile_base);

    auto digit_of = [&](KeyT k) -> uint32_t {
        if constexpr (BYTE_KEYS) return s_lut[k];
        else return (uint32_t)(k >> shift) & 0xFFu;
    };

    // ---- load (warp-striped: lane l, item k <-> tile offset warp*32*IPT + k*32 + l)
    KeyT key[IPT];
    uint32_t val[IPT];
    uint16_t rnk[IPT];
    const uint32_t wbase = warp * 32u * IPT + lane;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t local = wbase + k * 32u;
        const bool valid = local < nvalid;
        key[k] = valid ? kin[tile_base + local] : (KeyT)(~(KeyT)0);
        if (VAL_MODE == 1) val[k] = valid ? vin[tile_base + local] : 0u;
        if (VAL_MODE == 2) val[k] = tile_base + local;
    }

    // ---- rank inside the warp: match.any groups equal digits, the group's
    //      first lane bumps the warp's private counter.
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const bool valid = (wbase + k * 32u) < nvalid;
        const uint32_t d = valid ? digit_of(key[k]) : 255u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t leader = __ffs(peers) - 1;
        uint32_t before = 0;
        uint32_t *cnt = &s_whist[warp * RADIX + d];
        if (lane == leader) {
            before = *cnt;
            *cnt = before + __popc(peers);
        }
        before = __shfl_sync(0xffffffffu, before, leader);
        rnk[k] = (uint16_t)(before + __popc(peers & lanemask_lt()));
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit: exclusive prefix over warps, tile count, publish aggregate
    uint32_t bt = 0;
    if (tid < RADIX) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const uint32_t c = s_whist[w * RADIX + tid];
            s_whist[w * RADIX + tid] = run;
            run += c;
        }
        bt = run;
        st_volatile_u32(&lookback[(size_t)tile * RADIX + tid], (tile == 0 ? LB_INC : LB_AGG) | bt);
    }
    uint32_t wtotal;
    const uint32_t ex = warp_excl_sum(bt, wtotal);
    if (lane == 0) s_misc[1 + warp] = wtotal;
    __syncthreads();
    uint32_t wprefix = 0;
    for (uint32_t w = 0; w < warp; ++w) wprefix += s_misc[1 + w];
    const uint32_t bexcl = ex + wprefix;   // first slot of digit `tid` inside the sorted tile
    if (tid < RADIX) {
#pragma unroll
        for (int w = 0; w < WARPS; ++w) s_whist[w * RADIX + tid] += bexcl;
    }
    __syncthreads();

    // ---- stage keys in digit order
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const bool valid = (wbase + k * 32u) < nvalid;
        const uint32_t d = valid ? digit_of(key[k]) : 255u;
        const uint32_t slot = s_whist[warp * RADIX + d] + rnk[k];
        rnk[k] = (uint16_t)slot;
        s_keys[slot] = key[k];
    }

    // ---- decoupled look-back: exclusive count of this digit in earlier tiles
    if (tid < RADIX) {
        uint32_t excl = 0;
        if (tile > 0) {
            int64_t t = (int64_t)tile - 1;
            while (true) {
                const uint32_t v = ld_volatile_u32(&lookback[(size_t)t * RADIX + tid]);
                const uint32_t flag = v >> 30;
                if (flag == 0) continue;
                excl += v & LB_VAL;
                if (flag == 2) break;
                --t;
            }
            st_volatile_u32(&lookback[(size_t)tile * RADIX + tid], LB_INC | (excl + bt));
        }
        s_gbase[tid] = digit_base[tid] + excl - bexcl;
    }
    __syncthreads();

    // ---- coalesced write-out: consecutive threads take consecutive sorted slots
    uint32_t gpos[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t i = k * THREADS + tid;
        gpos[k] = 0;
        if (i < nvalid) {
            const KeyT kk = s_keys[i];
            gpos[k] = s_gbase[digit_of(kk)] + i;
            kout[gpos[k]] = kk;
        }
    }
    if (VAL_MODE != 0) {
        __syncthreads();
#pragma unroll
        for (int k = 0; k < IPT; ++k) s_vals[rnk[k]] = val[k];
        __syncthreads();
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const uint32_t i = k * THREADS + tid;
            if (i < nvalid) vout[gpos[k]] = s_vals[i];
        }
    }
}


// ---------------------------------------------------------------------------
// (uint64 key, uint32 value) pass, the K1 hot kernel.  512 threads, 4096 pairs
// per CTA, two CTAs per SM.  The tile is pulled into shared memory by the TMA
// engine (cp.async.bulk + mbarrier: no registers held while the 48 KB are in
// flight), ranked from shared memory, staged in digit order in a second
// shared buffer and written out as coalesced runs.
// ---------------------------------------------------------------------------
constexpr int OS_IPT = 8;            // default pairs per thread
#ifndef OS_LB_BATCH
#define OS_LB_BATCH 8
#endif
static_assert(SORT64_TILE >= 2048, "scratch sizing assumes tiles of at least 2048 pairs");

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// Shared memory of one CTA.  The TMA destination doubles as the digit-ordered staging buffer: by the
// time the tile is staged every thread holds its keys and values in registers.
template <int THREADS, int IPT = OS_IPT>
struct __align__(16) OsSmem {
    static constexpr int TILE = THREADS * IPT;
    static constexpr int WARPS = THREADS / 32;
    uint64_t keys[TILE];
    uint32_t vals[TILE];
    uint16_t whist[WARPS][RADIX];   // per-warp digit counters -> slots
    uint32_t gbase[RADIX];
    uint32_t wsum[32];
    uint32_t tile;
    uint64_t bar;
};

// lanes of the warp holding the same 8-bit digit: eight ballots, one per digit bit (fixed cost; match.any costs ~37
// ADU cycles at ~30 distinct digits per warp and only wins below ~8 distinct values).  Spelled in PTX -- test, vote,
// conditional complement, and: ptxas turns the eight bit tests of an item into one R2P, 3.2 instructions per digit
// bit where the C++ form (shift, and, two compares, select, and) compiles to six.
__device__ __forceinline__ uint32_t digit_peers(uint32_t d)
{
    uint32_t peers = 0xffffffffu;
#pragma unroll
    for (int bit = 0; bit < 8; ++bit) {
        uint32_t x;
        asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
                     "and.b32 t, %1, %2;\n\t"
                     "setp.ne.u32 p, t, 0;\n\t"
                     "vote.sync.ballot.b32 %0, p, 0xffffffff;\n\t"
                     "@!p not.b32 %0, %0;\n\t}"
                     : "=r"(x) : "r"(d), "r"(1u << bit));
        peers &= x;
    }
    return peers;
}

template <int THREADS, int MIN_CTAS, bool IDENT, int IPT = OS_IPT>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
onesweep64_kernel(const uint64_t *__restrict__ kin, uint64_t *__restrict__ kout, const uint32_t *__restrict__ vin,
                  uint32_t *__restrict__ vout, uint32_t n, int shift, const uint32_t *__restrict__ digit_base,
                  uint32_t *lookback, uint32_t *ticket, uint32_t *__restrict__ lookback_next)
{
    using Smem = OsSmem<THREADS, IPT>;
    constexpr int TILE = Smem::TILE;
    constexpr int WARPS = Smem::WARPS;
    static_assert(THREADS >= RADIX, "one thread per digit");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

    if (tid == 0) {
        S.tile = atomicAdd(ticket, 1u);
        mbar_init(&S.bar, 1);
    }
    for (int i = tid; i < WARPS * RADIX / 2; i += THREADS) reinterpret_cast<uint32_t *>(&S.whist[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint32_t tile_base = tile * (uint32_t)TILE;
    const uint32_t nvalid = min((uint32_t)TILE, n - tile_base);

    // the look-back rows of the NEXT pass (the other half of the table) are cleared here, tile by tile: no memset
    // launch between the passes
    if (tid < RADIX) lookback_next[(size_t)tile * RADIX + tid] = 0u;

    // ---- TMA: one thread arms the barrier and issues two bulk copies (16-byte granules);
    //      a ragged tail (last tile only) is finished with plain loads.
    const uint32_t nk16 = nvalid & ~1u;          // keys copied in 16-byte units
    const uint32_t nv16 = nvalid & ~3u;          // values copied in 16-byte units
    //      IDENT: the values are the identity (first pass over freshly packed keys) -- nothing to load.
    constexpr bool ident = IDENT;
    if (tid == 0) {
        mbar_expect_tx(&S.bar, nk16 * 8u + (ident ? 0u : nv16 * 4u));
        if (nk16) bulk_g2s(S.keys, kin + tile_base, nk16 * 8u, &S.bar);
        if (nv16 && !ident) bulk_g2s(S.vals, vin + tile_base, nv16 * 4u, &S.bar);
        if (nk16 < nvalid) S.keys[nk16] = kin[tile_base + nk16];                             // at most 1 key
    }
    if (!ident && tid < 4 && nv16 + tid < nvalid) S.vals[nv16 + tid] = vin[tile_base + nv16 + tid];    // at most 3 values
    mbar_wait(&S.bar, 0);
    __syncthreads();

    // ---- rank inside the warp (warp-striped: lane l, item k <-> tile offset warp*32*IPT + k*32 + l)
    //      Slots past the end of the array read as all-ones keys: digit 255 at every shift, ranked last.
    uint64_t key[IPT];
    uint32_t val[IPT];
    uint32_t peers[IPT];
    uint32_t dr[IPT];          // digit << 16 | rank of the item among the warp's items with that digit
    const uint32_t wbase = warp * 32u * IPT + lane;
    // all ballots first (they are independent), then the counter updates: batching the ballots by 8 to shorten the
    // live range of the peer masks was measured slower (0.649 vs 0.622 ms per pass at 512 x 16)
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t local = wbase + k * 32u;
        key[k] = (local < nvalid) ? S.keys[local] : ~0ULL;
        val[k] = ident ? tile_base + local : S.vals[local];
        const uint32_t d = (uint32_t)(key[k] >> shift) & 0xFFu;
        dr[k] = d << 16;
        peers[k] = digit_peers(d);
    }
    const uint32_t lt = lanemask_lt();
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        // the lowest lane of a digit group adds the group to the warp's counter; everybody reads the counter back
        // and takes its place from the end: rank = counter - #(peers at or above me)
        uint16_t *cnt = &S.whist[warp][dr[k] >> 16];
        const uint32_t np = __popc(peers[k]);
        if ((peers[k] & lt) == 0u) *cnt = (uint16_t)(*cnt + np);
        __syncwarp();
        dr[k] |= (uint32_t)*cnt - (uint32_t)__popc(peers[k] & ~lt);
        __syncwarp();
    }
    __syncthreads();     // every thread holds its keys/values: S.keys / S.vals may be overwritten below

    // ---- per digit: exclusive prefix over warps, tile count, publish the aggregate
    uint32_t bt = 0;
    if (tid < RADIX) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const uint32_t c = S.whist[w][tid];
            S.whist[w][tid] = (uint16_t)run;
            run += c;
        }
        bt = run;
        st_volatile_u32(&lookback[(size_t)tile * RADIX + tid], (tile == 0 ? LB_INC : LB_AGG) | bt);
    }
    uint32_t wtotal;
    const uint32_t ex = warp_excl_sum(bt, wtotal);
    if (lane == 0) S.wsum[warp] = wtotal;
    __syncthreads();
    uint32_t wprefix = 0;
    for (uint32_t w = 0; w < warp && w < RADIX / 32; ++w) wprefix += S.wsum[w];
    const uint32_t bexcl = ex + wprefix;          // first slot of digit `tid` inside the sorted tile
    if (tid < RADIX) {
#pragma unroll
        for (int w = 0; w < WARPS; ++w) S.whist[w][tid] = (uint16_t)(S.whist[w][tid] + bexcl);
    }
    __syncthreads();

    // ---- stage (key, value) in digit order
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t slot = (uint32_t)S.whist[warp][dr[k] >> 16] + (dr[k] & 0xFFFFu);
        S.keys[slot] = key[k];
        S.vals[slot] = val[k];
    }

    // ---- decoupled look-back, OS_LB_BATCH predecessors per round trip (8: measured best of 2 / 4 / 8; issuing
    //      the first batch before the staging stores was slower -- register pressure)
    if (tid < RADIX) {
        uint32_t excl = 0;
        if (tile > 0) {
            int64_t t = (int64_t)tile - 1;
            bool done = false;
            while (!done) {
                uint32_t v[OS_LB_BATCH];
#pragma unroll
                for (int j = 0; j < OS_LB_BATCH; ++j)
                    v[j] = (t - j >= 0) ? ld_volatile_u32(&lookback[(size_t)(t - j) * RADIX + tid]) : LB_INC;
#pragma unroll
                for (int j = 0; j < OS_LB_BATCH; ++j) {
                    if (done) break;
                    const uint32_t flag = v[j] >> 30;
                    if (flag == 0) break;             // not published yet: re-poll from here
                    excl += v[j] & LB_VAL;
                    --t;
                    if (flag == 2) done = true;
                }
            }
            st_volatile_u32(&lookback[(size_t)tile * RADIX + tid], LB_INC | (excl + bt));
        }
        S.gbase[tid] = digit_base[tid] + excl - bexcl;
    }
    __syncthreads();

    // ---- coalesced write-out: consecutive threads take consecutive sorted slots
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t i = k * THREADS + tid;
        if (i < nvalid) {
            const uint64_t kk = S.keys[i];
            const uint32_t g = S.gbase[(uint32_t)(kk >> shift) & 0xFFu] + i;
            kout[g] = kk;
            vout[g] = S.vals[i];
        }
    }
}

template <typename KeyT, int VAL_MODE, int THREADS, int IPT>
static constexpr size_t onesweep_smem()
{
    constexpr size_t fixed = (size_t)(THREADS / 32) * RADIX * 4 + RADIX * 4 + 64 * 4 + 256;
    constexpr size_t elem = (VAL_MODE != 0 && sizeof(KeyT) < 4) ? 4 : sizeof(KeyT);
    return fixed + elem * (size_t)THREADS * IPT;
}

// PASSES known at compile time: one uniformity test per key (runs of one key: all-same texts) instead of one per
// digit, the digits by shift + mask on the key's halves
template <int PASSES>
__global__ void __launch_bounds__(256)
radix_hist_kernel(const uint64_t *__restrict__ keys, uint32_t n, uint32_t *__restrict__ ghist)
{
    __shared__ uint32_t s_hist[8 * RADIX];
    hist_zero(s_hist, PASSES);
    __syncthreads();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const bool valid = i < n;
        const uint64_t key = valid ? keys[i] : 0ULL;
        hist_add_key_unsorted<PASSES>(s_hist, key, valid);
    }
    __syncthreads();
    hist_flush(s_hist, ghist, PASSES);
}

// block p: exclusive scan of hist[p][0..255] -> base[p][0..255]
__global__ void radix_scan_kernel(const uint32_t *__restrict__ hist, uint32_t *__restrict__ base)
{
    const uint32_t tid = threadIdx.x;
    uint32_t total;
    base[blockIdx.x * RADIX + tid] = block_excl_scan(hist[blockIdx.x * RADIX + tid], 0u, Plus(), total);
}

size_t sort_scratch_words(uint64_t n)
{
    const uint64_t tiles = (n + SORT64_TILE - 1) / SORT64_TILE + 1;
    return 8 * RADIX * 2 + 64 + 2 * tiles * RADIX + 256;
}

SortScratch carve_sort_scratch(Carver &c, uint64_t n)
{
    SortScratch s;
    const uint64_t tiles = (n + SORT64_TILE - 1) / SORT64_TILE + 1;
    s.hist = c.take<uint32_t>(8 * RADIX);
    s.base = c.take<uint32_t>(8 * RADIX);
    s.ticket = c.take<uint32_t>(64);
    s.lookback_words = 2 * tiles * RADIX;      // two halves, used by alternate passes of the (u64, u32) sort
    s.lookback = c.take<uint32_t>(s.lookback_words);
    return s;
}

cudaError_t radix_histogram_u64(const uint64_t *d_keys, uint32_t n, int passes, const SortScratch &s,
                                cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(s.hist, 0, 8 * RADIX * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    if (n == 0) return cudaSuccess;
    int blocks = (int)std::min<uint64_t>((n + 1023) / 1024, (uint64_t)num_sms() * 8);
    prof::Scope ps(st, prof::RADIX_SCAN, (uint64_t)n * 8);
    switch (passes) {
#define HK_HIST(P) case P: radix_hist_kernel<P><<<blocks, 256, 0, st>>>(d_keys, n, s.hist); break;
        HK_HIST(1) HK_HIST(2) HK_HIST(3) HK_HIST(4) HK_HIST(5) HK_HIST(6) HK_HIST(7)
        default: radix_hist_kernel<8><<<blocks, 256, 0, st>>>(d_keys, n, s.hist); break;
#undef HK_HIST
    }
    count_launch();
    return cudaGetLastError();
}

template <int THREADS, int MIN_CTAS, int IPT = OS_IPT>
static cudaError_t run_onesweep64(uint64_t *k0, uint32_t *v0, uint64_t *k1, uint32_t *v1, uint32_t n, int passes,
                                  const SortScratch &s, cudaStream_t st, bool identity_vals)
{
    using Smem = OsSmem<THREADS, IPT>;
    constexpr size_t smem = sizeof(Smem) + 128;
    auto kern = onesweep64_kernel<THREADS, MIN_CTAS, false, IPT>;
    auto kern_ident = onesweep64_kernel<THREADS, MIN_CTAS, true, IPT>;
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kern_ident, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_done = true;
    }
    const uint32_t tiles = (n + Smem::TILE - 1) / Smem::TILE;
    uint64_t *kin = k0, *kout = k1;
    uint32_t *vin = v0, *vout = v1;
    // the look-back table has two halves used by alternate passes; a pass clears the other half for its successor
    const size_t half = (size_t)tiles * RADIX;
    cudaError_t e = cudaMemsetAsync(s.lookback, 0, 2 * half * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    for (int p = 0; p < passes; ++p) {
        uint32_t *lb = s.lookback + (size_t)(p & 1) * half, *lb_next = s.lookback + (size_t)((p + 1) & 1) * half;
        {
            prof::Scope ps(st, prof::ONESWEEP_U64, (uint64_t)n * ((p == 0 && identity_vals) ? 20 : 24));
            if (p == 0 && identity_vals)
                kern_ident<<<tiles, THREADS, smem, st>>>(kin, kout, nullptr, vout, n, 0, s.base, lb, s.ticket, lb_next);
            else
                kern<<<tiles, THREADS, smem, st>>>(kin, kout, vin, vout, n, 8 * p, s.base + p * RADIX, lb,
                                                   s.ticket + p, lb_next);
            count_launch();
        }
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        uint64_t *tk = kin; kin = kout; kout = tk;
        uint32_t *tv = vin; vin = vout; vout = tv;
    }
    return cudaSuccess;
}

cudaError_t radix_sort_pairs_u64(uint64_t *k0, uint32_t *v0, uint64_t *k1, uint32_t *v1, uint32_t n,
                                 int passes, const SortScratch &s, cudaStream_t st, bool identity_vals)
{
    if (n == 0 || passes <= 0) return cudaSuccess;
    radix_scan_kernel<<<passes, RADIX, 0, st>>>(s.hist, s.base);
    count_launch();
    cudaError_t e = cudaMemsetAsync(s.ticket, 0, 64 * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    // ballots spelled in PTX; profiles/r01_onesweep_variants.txt keeps the numbers of the round-1 alternatives
    // (256 x 8 / 512 x 8, match.any ranking, C++ ballots, a persistent two-stage kernel)
#ifdef HKCSA_OS_SHAPES      // experiment build: tile shapes selectable at run time (tools/sort_probe.py)
    static int shape = -1;
    if (shape < 0) { const char *e = getenv("HKCSA_OS_SHAPE"); shape = e ? atoi(e) : 0; }
    switch (shape) {
        case 1: return run_onesweep64<256, 4, 12>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 2: return run_onesweep64<256, 3, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 3: return run_onesweep64<384, 2, 12>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 4: return run_onesweep64<512, 2, 12>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 5: return run_onesweep64<384, 4, 6>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 6: return run_onesweep64<256, 5, 8>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 7: return run_onesweep64<320, 4, 8>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 8: return run_onesweep64<256, 2, 24>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 9: return run_onesweep64<256, 3, 20>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 10: return run_onesweep64<384, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 11: return run_onesweep64<512, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 12: return run_onesweep64<512, 1, 24>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 13: return run_onesweep64<256, 4, 14>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 14: return run_onesweep64<256, 2, 32>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 15: return run_onesweep64<320, 3, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 16: return run_onesweep64<448, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 17: return run_onesweep64<512, 2, 12>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 18: return run_onesweep64<1024, 1, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 19: return run_onesweep64<768, 1, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 20: return run_onesweep64<480, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 21: return run_onesweep64<416, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 22: return run_onesweep64<448, 2, 18>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        case 23: return run_onesweep64<384, 2, 20>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
        default: break;
    }
#endif
    // Large arrays: 448 threads x 16 pairs = 7168 pairs per tile, 2 CTAs per SM -- the per-tile work (256-digit prefix
    // over the warps, look-back, five block barriers) is spread over 2.3x the pairs of the 384 x 8 tile: 0.621 vs 0.720 ms
    // per pass of 10^8 pairs (profiles/r02_onesweep_shapes.txt; 512 x 16: 0.627, 384 x 16: 0.638, 256 x 16 x 3 CTAs: 0.648,
    // 256 x 24: 0.638, 20+ pairs per thread: slower).  Small arrays keep the 3072-pair tile so that every SM gets tiles.
    if (n >= (1u << 22)) return run_onesweep64<448, 2, 16>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
    return run_onesweep64<384, 3>(k0, v0, k1, v1, n, passes, s, st, identity_vals);
}

cudaError_t radix_partition_bytes(const uint8_t *d_in, uint8_t *d_out, uint32_t *d_pos_out, uint32_t n,
                                  const uint8_t *d_lut, const uint32_t *d_bucket_base,
                                  const SortScratch &s, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const uint32_t tiles = (n + SORT8_TILE - 1) / SORT8_TILE;
    cudaError_t e = cudaMemsetAsync(s.ticket, 0, 64 * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(s.lookback, 0, (size_t)tiles * RADIX * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    if (d_pos_out) {
        constexpr size_t smem = onesweep_smem<uint8_t, 2, SORT8_THREADS, SORT8_IPT>();
        auto kern = onesweep_kernel<uint8_t, 2, SORT8_THREADS, SORT8_IPT>;
        static bool attr_done = false;
        if (!attr_done) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            attr_done = true;
        }
        kern<<<tiles, SORT8_THREADS, smem, st>>>(d_in, d_out, nullptr, d_pos_out, n, 0, d_lut, d_bucket_base,
                                                 s.lookback, s.ticket);
    } else {
        constexpr size_t smem = onesweep_smem<uint8_t, 0, SORT8_THREADS, SORT8_IPT>();
        auto kern = onesweep_kernel<uint8_t, 0, SORT8_THREADS, SORT8_IPT>;
        kern<<<tiles, SORT8_THREADS, smem, st>>>(d_in, d_out, nullptr, nullptr, n, 0, d_lut, d_bucket_base,
                                                 s.lookback, s.ticket);
    }
    count_launch();
    return cudaGetLastError();
}

}  // namespace hkcsa

// ------------------------------------------------------------------ C-ABI
using namespace hkcsa;

extern "C" size_t hkcsa_sort_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    carve_sort_scratch(c, n);
    return c.total();
}

extern "C" int hkcsa_sort_pairs_u64(uint64_t *d_keys, uint32_t *d_vals, uint64_t *d_keys_alt,
                                    uint32_t *d_vals_alt, uint64_t n, int key_bits, void *d_scratch,
                                    size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    HK_REQUIRE(key_bits >= 0 && key_bits <= 64, HKCSA_EINVAL, "key_bits must be in [0,64]");
    if (n == 0 || key_bits == 0) return HKCSA_OK;
    HK_REQUIRE(d_keys && d_vals && d_keys_alt && d_vals_alt && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(((reinterpret_cast<uintptr_t>(d_keys) | reinterpret_cast<uintptr_t>(d_vals) |
                 reinterpret_cast<uintptr_t>(d_keys_alt) | reinterpret_cast<uintptr_t>(d_vals_alt)) & 15) == 0,
               HKCSA_EINVAL, "sort buffers must be 16-byte aligned (TMA bulk copies)");
    Carver c(d_scratch);
    SortScratch s = carve_sort_scratch(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "sort scratch too small");
    cudaStream_t st = as_stream(stream);
    const int passes = (key_bits + 7) / 8;
    HK_CUDA(radix_histogram_u64(d_keys, (uint32_t)n, passes, s, st));
    HK_CUDA(radix_sort_pairs_u64(d_keys, d_vals, d_keys_alt, d_vals_alt, (uint32_t)n, passes, s, st));
    if (passes & 1) {
        HK_CUDA(cudaMemcpyAsync(d_keys, d_keys_alt, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
        HK_CUDA(cudaMemcpyAsync(d_vals, d_vals_alt, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    }
    return HKCSA_OK;
}
