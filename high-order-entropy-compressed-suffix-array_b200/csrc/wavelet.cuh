// wavelet.cuh -- device-side view of the level-wise wavelet tree (K3) shared by
// the build kernels (wavelet.cu) and the FM search kernels (fm_search.cu).
#pragma once
#include "common.cuh"
#include <type_traits>

namespace hkcsa {

constexpr uint32_t NODE_BIT_FLAG = 1u << 31;   // node_start's top bit = the bit a code takes at that level
constexpr uint32_t NODE_START_MASK = NODE_BIT_FLAG - 1u;

// Resident in the index blob at plan.off_tables.
struct WtTables {
    uint16_t code_of_sym[256];                  // byte -> dense code, 0xFFFF = absent
    uint8_t sym_of_code[256];
    uint8_t depth[256];                         // levels a code takes part in
    uint32_t C[260];                            // C[code] (+ total at [sigma])
    uint32_t node_start[HKCSA_MAX_LEVELS][256]; // per (level, code): start of the code's node | bit << 31
    uint32_t node_ones[HKCSA_MAX_LEVELS][256];  // rank1(level, node start)
    // build-time tables (wt_levels_kernel)
    uint8_t code8_of_sym[256];                  // byte -> dense code (present symbols only)
    uint8_t node_lo[HKCSA_MAX_LEVELS][256];     // per (level, code): first code of the code's node
    uint8_t node_hi1[HKCSA_MAX_LEVELS][256];    // per (level, code): last code of the code's node
    uint8_t lvl_lo[HKCSA_MAX_LEVELS][128];      // per (level, node k): first code
    uint8_t lvl_hi1[HKCSA_MAX_LEVELS][128];     // per (level, node k): last code
    uint32_t lvl_nodes[HKCSA_MAX_LEVELS];
    // root-to-leaf paths: bit 7 - l of a path = the bit the symbol takes at level l, zeros below its leaf.  Paths order
    // like the codes, the level-l node of a symbol is the top l bits of its path.
    uint8_t path_of_sym[256];                   // byte -> path (present symbols only)
    uint16_t path_of_code[260];                 // [sigma] = 256
    uint16_t code_of_path[256];                 // 0xFFFF: no symbol has this path
};

// What one LF step reads at row j of a rank source: the code of bwt[j], its byte, and occ(code, j).
struct LfStep {
    uint32_t code, sym, occ;
};

// Shared-memory copy of what a symbol-rank walk needs ("C[] held in shared memory").
struct WtSmem {
    uint32_t node_start[HKCSA_MAX_LEVELS][256];
    uint32_t node_ones[HKCSA_MAX_LEVELS][256];
    uint32_t C[260];
    uint16_t code_of_sym[256];
    uint8_t depth[256];
    uint8_t sym_of_code[256];
};

// The tree as seen by device code; also the wavelet-tree rank source of the query kernels (fm_search.cu, extract.cu),
// which use load / rank2 / step with the tables in shared memory.
struct WtDev {
    const WtTables *tab;
    BitVec level[HKCSA_MAX_LEVELS];
    uint32_t levels;
    uint32_t sigma;
    uint64_t n;

    using Smem = WtSmem;
    using Row = uint32_t;
    __device__ void load(WtSmem &s) const;
    __device__ void rank2(const WtSmem &s, uint32_t code, uint32_t ch, uint32_t &a, uint32_t &b) const;
    __device__ LfStep step(const WtSmem &s, uint32_t j) const;
    // the plain LF step of extract: LF(j) = C[code] + occ (the walk is exact when the sentinel is unique)
    __device__ uint32_t next(const WtSmem &s, const LfStep &t, uint32_t) const { return s.C[t.code] + t.occ; }
};

static inline uint64_t rank_blocks_for(uint64_t bits) { return bits / HKCSA_BLOCK_BITS + 1; }
static inline uint64_t super_for(uint64_t bits) { return rank_blocks_for(bits) / HKCSA_SUPER_BLOCKS + 1; }
static inline uint64_t select_samples_for(uint64_t bits) { return bits / HKCSA_SELECT_SAMPLE + 2; }

static inline WtDev make_wt_dev(const void *d_blob, const hkcsa_wt_plan *p)
{
    WtDev d;
    const uint8_t *base = static_cast<const uint8_t *>(d_blob);
    d.tab = reinterpret_cast<const WtTables *>(base + p->off_tables);
    for (uint32_t l = 0; l < HKCSA_MAX_LEVELS; ++l) {
        d.level[l].blocks = reinterpret_cast<const RankBlock *>(base + p->off_blocks[l]);
        d.level[l].super = reinterpret_cast<const uint64_t *>(base + p->off_super[l]);
        d.level[l].len = p->level_len[l];
    }
    d.levels = p->levels;
    d.sigma = p->sigma;
    d.n = p->n;
    return d;
}

// Tile histogram + per-symbol exclusive prefix over tiles (wavelet.cu); also used by the sampled Occ table.
constexpr int WTL_THREADS = 256;
constexpr int WTL_TILE = 8192;
__global__ void __launch_bounds__(WTL_THREADS)
wt_tile_hist_kernel(const uint8_t *__restrict__ sym, uint64_t n, const WtTables *__restrict__ tab, uint32_t sigma,
                    uint32_t tiles, uint32_t *__restrict__ gcnt /* [sigma][tiles+1] */);
__global__ void __launch_bounds__(1024) wt_tile_scan_kernel(uint32_t *__restrict__ gcnt, uint32_t tiles);

// Where a count kernel puts its answers.  n == 0: the caller's own lo / hi arrays.  n > 0 (multi-GPU, patterns
// sharded): every rank's kernel writes its slice straight into the result arrays of ALL ranks through
// peer-mapped pointers (NVLink stores from inside the search kernel) at [base + pattern]: the all-gather of
// the results is fused into the search, there is no collective afterwards.
struct PeerOut {
    int64_t *lo[HKCSA_MAX_PEERS];
    int64_t *hi[HKCSA_MAX_PEERS];
    uint64_t base;
    uint32_t n;
};
template <bool PEERS>
__device__ __forceinline__ void put_range(const PeerOut &po, int64_t *out_lo, int64_t *out_hi, int64_t p, int64_t l, int64_t h)
{
    if (!PEERS) {
        out_lo[p] = l;
        out_hi[p] = h;
    } else {
        for (uint32_t r = 0; r < po.n; ++r) {
            po.lo[r][po.base + p] = l;
            po.hi[r][po.base + p] = h;
        }
    }
}

__device__ __forceinline__ void wt_smem_load(WtSmem &s, const WtDev &wt)
{
    const WtTables *t = wt.tab;
    for (uint32_t i = threadIdx.x; i < wt.levels * 256u; i += blockDim.x) {
        (&s.node_start[0][0])[i] = (&t->node_start[0][0])[i];
        (&s.node_ones[0][0])[i] = (&t->node_ones[0][0])[i];
    }
    for (uint32_t i = threadIdx.x; i < 260u; i += blockDim.x) s.C[i] = t->C[i];
    for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) {
        s.code_of_sym[i] = t->code_of_sym[i];
        s.depth[i] = t->depth[i];
        s.sym_of_code[i] = t->sym_of_code[i];
    }
}

// Reads of the descent tables: WtSmem is in shared memory; WtTables is the copy in global memory (the sliced index
// of MsDev, multi_slice.cuh), read through the read-only path.
template <typename Tab, typename T>
__device__ __forceinline__ T wt_ld(const T &x)
{
    if constexpr (std::is_same_v<Tab, WtTables>) return __ldg(&x);
    else return x;
}

// occ(code, i) = occurrences of `code` in the sequence before position i.
template <typename Tab>
__device__ __forceinline__ uint32_t wt_rank_code(const Tab &t, const WtDev &wt, uint32_t code, uint32_t i)
{
    uint32_t p = i;
    const uint32_t dep = t.depth[code];
    for (uint32_t l = 0; l < dep; ++l) {
        const uint32_t ns = wt_ld<Tab>(t.node_start[l][code]);
        const uint32_t start = ns & NODE_START_MASK;
        const uint32_t r1 = (uint32_t)bv_rank(wt.level[l], (uint64_t)start + p) - wt_ld<Tab>(t.node_ones[l][code]);
        p = (ns & NODE_BIT_FLAG) ? r1 : (p - r1);
    }
    return p;
}

// Two positions of the same code at once (the l / r boundaries of a backward-
// search step): the loads of both walks are issued together.
__device__ __forceinline__ void wt_rank_code2(const WtSmem &s, const WtDev &wt, uint32_t code, uint32_t &a,
                                              uint32_t &b)
{
    const uint32_t dep = s.depth[code];
    for (uint32_t l = 0; l < dep; ++l) {
        const uint32_t ns = s.node_start[l][code];
        const uint32_t start = ns & NODE_START_MASK;
        const uint32_t ones0 = s.node_ones[l][code];
        const BitVec &v = wt.level[l];
        const uint64_t ia = (uint64_t)start + a, ib = (uint64_t)start + b;
        const uint64_t ba = ia / HKCSA_BLOCK_BITS, bb = ib / HKCSA_BLOCK_BITS;
        const RankBlock qa = load_block(v.blocks + ba);
        // once the range is narrow both boundaries fall into the same 224-bit block: one sector, not two
        const RankBlock qb = (bb == ba) ? qa : load_block(v.blocks + bb);
        const uint32_t ra = (uint32_t)(v.super[ba / HKCSA_SUPER_BLOCKS] + (uint32_t)(qa.w[0] & 0xFFFFFFFFu) +
                                       block_rank(qa, (uint32_t)(ia - ba * HKCSA_BLOCK_BITS))) - ones0;
        const uint32_t rb = (uint32_t)(v.super[bb / HKCSA_SUPER_BLOCKS] + (uint32_t)(qb.w[0] & 0xFFFFFFFFu) +
                                       block_rank(qb, (uint32_t)(ib - bb * HKCSA_BLOCK_BITS))) - ones0;
        if (ns & NODE_BIT_FLAG) { a = ra; b = rb; }
        else { a -= ra; b -= rb; }
    }
}

// access + rank in one descent: code at position i and occ(code, i).
template <typename Tab>
__device__ __forceinline__ uint32_t wt_access_rank(const Tab &t, const WtDev &wt, uint32_t i, uint32_t &occ)
{
    uint32_t lo = 0, hi = wt.sigma, p = i;
    for (uint32_t l = 0; hi - lo > 1; ++l) {
        const uint32_t mid = lo + (hi - lo) / 2;
        const uint32_t start = wt_ld<Tab>(t.node_start[l][lo]) & NODE_START_MASK;
        const BitVec &v = wt.level[l];
        const uint64_t ia = (uint64_t)start + p;
        const uint64_t ba = ia / HKCSA_BLOCK_BITS;
        const uint32_t o = (uint32_t)(ia - ba * HKCSA_BLOCK_BITS);
        const RankBlock q = load_block(v.blocks + ba);
        const uint32_t r1 = (uint32_t)(v.super[ba / HKCSA_SUPER_BLOCKS] + (uint32_t)(q.w[0] & 0xFFFFFFFFu) +
                                       block_rank(q, o)) - wt_ld<Tab>(t.node_ones[l][lo]);
        if (block_bit(q, o)) { p = r1; lo = mid; }
        else { p -= r1; hi = mid; }
    }
    occ = p;
    return lo;
}

__device__ __forceinline__ void WtDev::load(WtSmem &s) const { wt_smem_load(s, *this); }
// with one symbol the depth is 0: the descent keeps both boundaries
__device__ __forceinline__ void WtDev::rank2(const WtSmem &s, uint32_t code, uint32_t, uint32_t &a, uint32_t &b) const
{
    wt_rank_code2(s, *this, code, a, b);
}
__device__ __forceinline__ LfStep WtDev::step(const WtSmem &s, uint32_t j) const
{
    LfStep t;
    t.code = wt_access_rank(s, *this, j, t.occ);
    t.sym = s.sym_of_code[t.code];
    return t;
}

}  // namespace hkcsa
