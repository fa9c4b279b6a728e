// common.cuh -- shared helpers for libhkcsa (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <atomic>

#include "../../include/hkcsa.h"

namespace hkcsa {

// ---------------------------------------------------------------- errors
void set_error(const char *fmt, ...);

#define HK_CUDA(call)                                                                      \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            hkcsa::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,                  \
                             cudaGetErrorString(e__));                                     \
            return HKCSA_ECUDA;                                                            \
        }                                                                                  \
    } while (0)

// every kernel launch of the library is counted (bench.py reports gpu_launches)
extern std::atomic<unsigned long long> g_launches;
static inline void count_launch(unsigned long long k = 1) { g_launches.fetch_add(k, std::memory_order_relaxed); }

#define HK_LAUNCH_CHECK()                                                                  \
    do {                                                                                   \
        hkcsa::count_launch();                                                             \
        HK_CUDA(cudaGetLastError());                                                       \
    } while (0)

#define HK_REQUIRE(cond, code, msg)                                                        \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            hkcsa::set_error("%s:%d %s", __FILE__, __LINE__, msg);                         \
            return (code);                                                                 \
        }                                                                                  \
    } while (0)

// One pinned host page per calling thread for scalar read-backs (the library's only
// allocation).  Returns nullptr on failure (error already set).
void *pinned_page();   // 4096 bytes

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Carves aligned sub-buffers out of one caller-provided scratch allocation.
struct Carver {
    uint8_t *base;
    size_t used;
    explicit Carver(void *p) : base(static_cast<uint8_t *>(p)), used(0) {}
    template <typename T>
    T *take(size_t count)
    {
        used = align_up(used, 256);
        T *p = base ? reinterpret_cast<T *>(base + used) : nullptr;
        used += count * sizeof(T);
        return p;
    }
    size_t total() const { return align_up(used, 256); }
};

static inline uint32_t bits_for(uint64_t maxval)  // bits needed to represent values 0..maxval
{
    uint32_t b = 0;
    while (b < 64 && (maxval >> b) != 0) ++b;
    return b;
}

static inline int num_sms()
{
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

// ---------------------------------------------------------------- device helpers
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint32_t lanemask_lt()
{
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t *p, uint32_t v)
{
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// L2 eviction policies (createpolicy, sm_80+): streams that are touched once are marked evict-first so they do
// not push a randomly gathered table (the text under the BWT gather) out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_policy_evict_last(float fraction = 1.0f)
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, %1;" : "=l"(p) : "f"(fraction));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint32_t ld_u8_hint(const uint8_t *p, uint64_t pol)
{
    uint32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ uint4 ld_u32x4_hint(const uint32_t *p, uint64_t pol)
{
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_u32_hint(uint32_t *p, uint32_t v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}

// Exclusive warp scan (sum) of one uint32 per lane.
__device__ __forceinline__ uint32_t warp_excl_sum(uint32_t v, uint32_t &total)
{
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane_id() >= (uint32_t)o) x += y;
    }
    total = __shfl_sync(0xffffffffu, x, 31);
    return x - v;
}
__device__ __forceinline__ uint32_t warp_incl_max(uint32_t v)
{
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane_id() >= (uint32_t)o) x = max(x, y);
    }
    return x;
}

// ---------------------------------------------------------------- CTA-wide scans
// Exclusive scans over one CTA (blockDim.x a multiple of 32) under an associative operator `op` with identity `id`.
// The operator is applied in order, prefix ⊕ value, so it need not commute.  Every thread of the CTA calls them.
template <typename T>
__device__ __forceinline__ T shfl_up(T v, uint32_t o)
{
    static_assert(sizeof(T) % 4 == 0, "shuffled in 32-bit words");
    uint32_t w[sizeof(T) / 4];
    memcpy(w, &v, sizeof(T));
#pragma unroll
    for (uint32_t i = 0; i < sizeof(T) / 4; ++i) w[i] = __shfl_up_sync(0xffffffffu, w[i], o);
    memcpy(&v, w, sizeof(T));
    return v;
}

// the prefix of this thread's v over the CTA; total = the whole CTA's.  Ends on a barrier, so it may be called again.
template <typename T, typename Op>
__device__ __forceinline__ T block_excl_scan(T v, T id, Op op, T &total)
{
    __shared__ T s_warp[32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    T x = v;
#pragma unroll
    for (uint32_t o = 1; o < 32; o <<= 1) {
        const T y = shfl_up(x, o);
        if (lane >= o) x = op(y, x);
    }
    const T before = shfl_up(x, 1);                  // inclusive prefix of the lane before
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {                                 // inclusive prefixes over the warps
        T w = lane < (blockDim.x >> 5) ? s_warp[lane] : id;
#pragma unroll
        for (uint32_t o = 1; o < 32; o <<= 1) {
            const T y = shfl_up(w, o);
            if (lane >= o) w = op(y, w);
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    total = s_warp[(blockDim.x >> 5) - 1];
    const T pre = warp ? s_warp[warp - 1] : id;
    __syncthreads();
    return lane ? op(pre, before) : pre;
}

// The same scan over `count` values in rounds of blockDim.x, carried from round to round: load(i) gives value i,
// store(i, p) takes its exclusive prefix.  Returns the total of all `count` values.
template <typename T, typename N, typename Op, typename Load, typename Store>
__device__ __forceinline__ T block_excl_scan_carried(N count, T id, Op op, Load load, Store store)
{
    T carry = id;
    for (N base = 0; base < count; base += blockDim.x) {
        const N i = base + threadIdx.x;
        T total;
        const T ex = block_excl_scan(i < count ? load(i) : id, id, op, total);
        if (i < count) store(i, op(carry, ex));
        carry = op(carry, total);
    }
    return carry;
}

struct Plus {
    template <typename T>
    __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};

// ---------------------------------------------------------------- rank blocks
// One 32-byte block: low 32 bits of word 0 = ones before the block (relative to
// its superblock); the other 224 bits are payload.  See include/hkcsa.h.
struct __align__(32) RankBlock {
    uint64_t w[4];
};

// ones among payload bits [0, o) of a block, o in [0, 224]
__device__ __forceinline__ uint32_t block_rank(const RankBlock &b, uint32_t o)
{
    const uint32_t t = o + 32u;         // bit index inside the 256-bit block
    const uint32_t wq = t >> 6, r = t & 63u;
    const uint64_t part = (r ? ((1ULL << r) - 1ULL) : 0ULL);
    uint64_t w0 = b.w[0] & 0xFFFFFFFF00000000ULL;
    uint32_t c = 0;
    c += __popcll(wq > 0 ? w0 : (w0 & part));
    c += __popcll(wq > 1 ? b.w[1] : (wq == 1 ? (b.w[1] & part) : 0ULL));
    c += __popcll(wq > 2 ? b.w[2] : (wq == 2 ? (b.w[2] & part) : 0ULL));
    c += __popcll(wq > 3 ? b.w[3] : (wq == 3 ? (b.w[3] & part) : 0ULL));
    return c;
}
__device__ __forceinline__ uint32_t block_bit(const RankBlock &b, uint32_t o)
{
    const uint32_t t = o + 32u;
    return (uint32_t)(b.w[t >> 6] >> (t & 63u)) & 1u;
}
// The exact LF step of locate: LF(j) = C[code] + lf_fix(occ(code, j), ...).  Row row0 holds suffix 0, whose BWT
// symbol c0 = text[n-1] stands for the one-symbol suffix n-1: the first of the c0-suffixes.  When c0 also occurs
// before row0 (a text that holds its last symbol elsewhere, e.g. a second '$'), occ alone ranks row0 after those
// rows: the true step is C[c0] at row0 and one more than occ on every c0-row before it.  fix = occ(c0, row0) != 0;
// with a unique sentinel it is 0 and the step is the plain one.
__device__ __forceinline__ uint32_t lf_fix(uint32_t occ, uint32_t code, uint32_t j, uint32_t c0, uint32_t row0,
                                           uint32_t fix)
{
    if (!fix || code != c0 || j > row0) return occ;
    return j == row0 ? 0u : occ + 1u;
}
// the same step over 64-bit rows (MsDev, the sliced index of the distributed build: multi_slice.cuh)
__device__ __forceinline__ uint64_t lf_fix(uint64_t occ, uint32_t code, uint64_t j, uint32_t c0, uint64_t row0,
                                           uint32_t fix)
{
    if (!fix || code != c0 || j > row0) return occ;
    return j == row0 ? 0ull : occ + 1ull;
}
// one 256-bit read-only load (sm_100: LDG.E.256) of a 32-byte-aligned sector
__device__ __forceinline__ void ld_nc_256(const void *p, uint64_t &w0, uint64_t &w1, uint64_t &w2, uint64_t &w3)
{
    asm("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(w0), "=l"(w1), "=l"(w2), "=l"(w3) : "l"(p));
}
__device__ __forceinline__ RankBlock load_block(const RankBlock *p)
{
    RankBlock b;          // the whole block = one sector = one load instruction
    ld_nc_256(p, b.w[0], b.w[1], b.w[2], b.w[3]);
    return b;
}

// A level bit-vector as seen by device code.
struct BitVec {
    const RankBlock *blocks;
    const uint64_t *super;   // absolute ones before each superblock
    uint64_t len;            // bits
};

// rank1(i) = ones in bits [0, i), i in [0, len]
__device__ __forceinline__ uint64_t bv_rank(const BitVec &v, uint64_t i)
{
    const uint64_t blk = i / HKCSA_BLOCK_BITS;
    const uint32_t o = (uint32_t)(i - blk * HKCSA_BLOCK_BITS);
    const RankBlock b = load_block(v.blocks + blk);
    return v.super[blk / HKCSA_SUPER_BLOCKS] + (uint32_t)(b.w[0] & 0xFFFFFFFFu) + block_rank(b, o);
}

// The mark test of a locate walk: is row j marked in the sampled SA, and if so slot = rank1(marks, j), the index of
// its sample.
__device__ __forceinline__ bool marked_slot(const BitVec &marks, uint32_t j, uint64_t &slot)
{
    const uint64_t g = j / HKCSA_BLOCK_BITS;
    const uint32_t o = j - (uint32_t)g * HKCSA_BLOCK_BITS;
    const RankBlock b = load_block(marks.blocks + g);
    if (!block_bit(b, o)) return false;
    slot = marks.super[g / HKCSA_SUPER_BLOCKS] + (uint32_t)(b.w[0] & 0xFFFFFFFFu) + block_rank(b, o);
    return true;
}

}  // namespace hkcsa
