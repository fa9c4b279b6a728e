// wavelet.cu -- K3: level-wise wavelet tree over the BWT with interleaved rank
// blocks, superblocks and select samples; bit-vector and symbol-level queries.
//
// Replaces WaveletTree.build_tree (reference csa/wavelet_tree.py:72-100),
// SuccinctRankSelect (:5-25) and, through rank-by-symbol, build_occ
// (utils/utils.py:26-32).  Tree shape = the reference's alphabet halving:
// node [lo,hi) over the sorted alphabet splits at mid = lo + (hi-lo)/2
// (:78-80); bit = 1 for symbols in the right half (:82).  The reference keeps
// the left-most node per level (:92,:99-100); we keep every node, laid out
// level by level in alphabet order, so its node is the prefix of each level.
#include "common.cuh"
#include "prof.cuh"
#include "radix_sort.cuh"
#include "wavelet.cuh"

namespace hkcsa {

constexpr int WTP_THREADS = 256;
constexpr int WTP_BLOCKS_PER_CTA = 64;                                   // rank blocks per CTA
constexpr int WTP_SYMS = WTP_BLOCKS_PER_CTA * (int)HKCSA_BLOCK_BITS;     // 14336 symbols per CTA

// Stores a tile of WTP_BLOCKS_PER_CTA rank blocks from its 448 payload words in shared memory, 7 per block: threads
// 0..63 write one block each, whose header is the count of ones before the block INSIDE the tile; the tile's ones go
// to agg[tile].
__device__ __forceinline__ void dir_store_tile(const uint32_t *s_words, RankBlock *__restrict__ blocks, uint64_t nblocks,
                                               uint32_t tile, uint32_t *__restrict__ agg)
{
    __shared__ uint32_t s_wsum[2];
    const uint32_t tid = threadIdx.x;
    const uint64_t gb = (uint64_t)tile * WTP_BLOCKS_PER_CTA + tid;
    uint32_t w[7] = {0, 0, 0, 0, 0, 0, 0};
    uint32_t cnt = 0;
    if (tid < WTP_BLOCKS_PER_CTA) {
#pragma unroll
        for (int t = 0; t < 7; ++t) { w[t] = s_words[tid * 7 + t]; cnt += __popc(w[t]); }
    }
    uint32_t wtot;
    const uint32_t ex = warp_excl_sum(cnt, wtot);
    if ((tid & 31u) == 31u && tid < WTP_BLOCKS_PER_CTA) s_wsum[tid >> 5] = wtot;
    __syncthreads();
    if (tid < WTP_BLOCKS_PER_CTA) {
        const uint32_t rel = ex + ((tid >= 32) ? s_wsum[0] : 0u);
        if (gb < nblocks) {
            uint4 *dst = reinterpret_cast<uint4 *>(blocks + gb);
            dst[0] = make_uint4(rel, w[0], w[1], w[2]);
            dst[1] = make_uint4(w[3], w[4], w[5], w[6]);
        }
        if (tid == WTP_BLOCKS_PER_CTA - 1) agg[tile] = rel + cnt;
    }
}

// Packs one level: bit j = lut_bit[sym[j]]; a tile of rank blocks per CTA (dir_store_tile).
__global__ void __launch_bounds__(WTP_THREADS)
wt_pack_kernel(const uint8_t *__restrict__ sym, uint64_t len, const uint8_t *__restrict__ lut_bit,
               RankBlock *__restrict__ blocks, uint64_t nblocks, uint32_t *__restrict__ agg)
{
    __shared__ uint8_t s_lut[256];
    __shared__ __align__(16) uint8_t s_bits[WTP_SYMS / 8];   // 1792 bytes, 28 per rank block
    const uint32_t tid = threadIdx.x;
    s_lut[tid] = lut_bit[tid];
    __syncthreads();
    const uint64_t sym_base = (uint64_t)blockIdx.x * WTP_SYMS;
    for (uint32_t q = tid; q < WTP_SYMS / 8; q += WTP_THREADS) {
        const uint64_t g = sym_base + (uint64_t)q * 8;
        uint32_t byte = 0;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const uint64_t j = g + t;
            const uint32_t bit = (j < len) ? s_lut[sym[j]] : 0u;
            byte |= bit << t;
        }
        s_bits[q] = (uint8_t)byte;
    }
    __syncthreads();
    dir_store_tile(reinterpret_cast<const uint32_t *>(s_bits), blocks, nblocks, blockIdx.x, agg);
}

// position (0-based, within the 224 payload bits) of the r-th one (r >= 1) of a block
__device__ __forceinline__ uint32_t block_select(const RankBlock &b, uint32_t r)
{
    uint64_t w[4] = {b.w[0] & 0xFFFFFFFF00000000ULL, b.w[1], b.w[2], b.w[3]};
    uint32_t base = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t c = __popcll(w[q]);
        if (r <= c) {
            uint64_t x = w[q];
            for (uint32_t k = 1; k < r; ++k) x &= x - 1;   // clear the r-1 lowest ones
            return base + (uint32_t)(__ffsll((long long)x) - 1) - 32u;
        }
        r -= c;
        base += 64;
    }
    return HKCSA_BLOCK_BITS;   // not found
}

struct BlockOnes {
    uint64_t before;   // ones before the block
    uint32_t in;       // ones in the block
};

// Finishes rank block g (contents b) of a level whose header still counts the ones before the block inside its tile
// of TILE blocks; carry[t] = ones before tile t of the level.  The header becomes relative to the block's superblock,
// a superblock that starts at g gets its count, and the select sample whose one falls in the block gets its position.
template <uint32_t TILE>
__device__ __forceinline__ BlockOnes dir_finish_block(const RankBlock &b, uint64_t g, RankBlock *__restrict__ blocks,
                                                      const uint64_t *__restrict__ carry, uint64_t *__restrict__ super,
                                                      uint32_t *__restrict__ select_samples)
{
    static_assert(HKCSA_SUPER_BLOCKS % TILE == 0, "superblocks must start on a tile");
    const uint32_t rel = (uint32_t)(b.w[0] & 0xFFFFFFFFu);
    const uint64_t before = carry[g / TILE] + rel;
    const uint64_t sb = g / HKCSA_SUPER_BLOCKS;
    const uint64_t sb_abs = carry[sb * (HKCSA_SUPER_BLOCKS / TILE)];
    reinterpret_cast<uint32_t *>(blocks + g)[0] = (uint32_t)(before - sb_abs);
    if (g % HKCSA_SUPER_BLOCKS == 0) super[sb] = sb_abs;
    const uint32_t cnt = block_rank(b, HKCSA_BLOCK_BITS);
    if (cnt) {
        // ones numbered before+1 .. before+cnt; sample t marks one number 1 + t*SAMPLE
        const uint64_t t = (before + HKCSA_SELECT_SAMPLE - 1) / HKCSA_SELECT_SAMPLE;
        const uint64_t k = 1 + t * HKCSA_SELECT_SAMPLE;
        if (k <= before + cnt) {
            const uint32_t bit = block_select(b, (uint32_t)(k - before));
            select_samples[t] = (uint32_t)(g * HKCSA_BLOCK_BITS + bit);
        }
    }
    return BlockOnes{before, cnt};
}

// ---------------------------------------------------------------- all levels in one sweep
// The sequence is cut into tiles of WTL_TILE symbols.  (1) wt_tile_hist: symbol counts per tile.
// (2) wt_tile_scan: per symbol, exclusive prefix over tiles.  (3) wt_levels: each CTA keeps its
// tile in shared memory and walks down the tree: at level l the tile is ordered by level-l node
// (stable), so the elements of one node are a contiguous run whose destination in the level's
// bit-vector is also contiguous: node start + (elements of that node in earlier tiles).  The run's
// bits are funnel-shifted to the destination word alignment and stored (whole words) or OR-ed
// (edge words shared with neighbouring tiles).  The next level's order is a stable split of every
// run by its bit, computed from a tile-wide prefix sum of the bits.  The sequence is read from HBM
// once for all levels and only bits are written.
constexpr int WTL_EPT = WTL_TILE / WTL_THREADS;   // 32 symbols per thread = one bit word
// resident CTAs per SM asked of the compiler for wt_levels_kernel: 77 registers gave 3 (C3: 3.41 ms), 4 CTAs 3.04 ms,
// 5 CTAs (47 registers, no spills) 2.63 ms, 6 CTAs 2.73 ms
#define WTL_MIN_CTAS 5
static_assert(WTL_EPT == 32, "one 32-bit word of bits per thread");

__global__ void __launch_bounds__(WTL_THREADS)
wt_tile_hist_kernel(const uint8_t *__restrict__ sym, uint64_t n, const WtTables *__restrict__ tab, uint32_t sigma,
                    uint32_t tiles, uint32_t *__restrict__ gcnt /* [sigma][tiles+1] */)
{
    __shared__ uint32_t s_h[256];
    __shared__ uint8_t s_code[256];
    const uint32_t tid = threadIdx.x;
    s_h[tid] = 0;
    s_code[tid] = tab->code8_of_sym[tid];
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * WTL_TILE;
    const uint32_t nv = (uint32_t)min((uint64_t)WTL_TILE, n - base);
    for (uint32_t i = tid; i < nv; i += WTL_THREADS) atomicAdd(&s_h[s_code[sym[base + i]]], 1u);
    __syncthreads();
    if (tid < sigma) gcnt[(size_t)tid * (tiles + 1) + blockIdx.x] = s_h[tid];
}

// one CTA per symbol: in-place exclusive scan of its tiles+1 entries (the last becomes the total)
__global__ void __launch_bounds__(1024)
wt_tile_scan_kernel(uint32_t *__restrict__ gcnt, uint32_t tiles)
{
    uint32_t *row = gcnt + (size_t)blockIdx.x * (tiles + 1);
    block_excl_scan_carried(tiles + 1, 0u, Plus(), [&](uint32_t t) { return t < tiles ? row[t] : 0u; },
                            [&](uint32_t t, uint32_t p) { row[t] = p; });
}

struct LevelWords {
    uint32_t *w[HKCSA_MAX_LEVELS];   // rank blocks of each level viewed as uint32[8] per block
};

// The CTA's tile as root-to-leaf PATHS (WtTables::path_of_sym), one byte per element: the bit of an element at level l
// is bit 7 - l of its path and its node is the top l bits, so the level loop needs no table look-up per element.  At
// level l the tile is ordered by the top l path bits (stable); the elements sharing them are one contiguous run
// [S, E) -- an internal node, or a leaf reached earlier whose remaining path bits are zero, so that splitting it moves
// nothing.  Per level:
//   A  bits: warp w owns tile positions [1024 w, 1024 w + 1024) as 32 rows of 32; one ballot per row gives the row's
//      word of bits (lane r of the warp keeps row r's word); ones before every row by a block scan of the popcounts;
//   B  emit: each internal node's run of bits goes to its place in the level's bit-vector (funnel-shifted to the
//      destination alignment; whole words stored, edge words OR-ed);
//   C  split: per run one table entry {split point M - ones before the run, ones before the run}; an element moves to
//      M + (ones before it inside the run) or to its position minus that count.  The lanes of a row read the same
//      entry (broadcast) and write two consecutive byte streams: no bank conflicts to speak of.
// Slots past the end of the text hold path 0xFF: they stay at the tail of the last run on every level and are never
// emitted (the runs' lengths come from the tile histogram, which does not count them).
__global__ void __launch_bounds__(WTL_THREADS, WTL_MIN_CTAS)
wt_levels_kernel(const uint8_t *__restrict__ sym, uint64_t n, const WtTables *__restrict__ tab,
                 const uint32_t *__restrict__ gpre, uint32_t tiles, LevelWords lv, uint32_t levels, uint32_t sigma)
{
    __shared__ __align__(16) uint8_t s_a[WTL_TILE];
    __shared__ __align__(16) uint8_t s_b[WTL_TILE];
    __shared__ uint2 s_wp[WTL_THREADS + 1];           // row r: .x = bits of tile positions [32 r, 32 r + 32), .y = ones before them
    __shared__ uint32_t s_tcum[257], s_gcum[257];     // per path x: elements with a smaller path in this tile / in earlier tiles
    __shared__ uint32_t s_ent[128];
    __shared__ uint8_t s_path[256];
    __shared__ uint32_t s_scan[2][8];

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;
    const uint64_t base = (uint64_t)tile * WTL_TILE;
    const uint32_t nv = (uint32_t)min((uint64_t)WTL_TILE, n - base);

    s_path[tid] = tab->path_of_sym[tid];
    {
        uint32_t cnt = 0, pre = 0;
        const uint32_t c = tab->code_of_path[tid];
        if (c < sigma) {
            const uint32_t *row = gpre + (size_t)c * (tiles + 1);
            pre = row[tile];
            cnt = row[tile + 1] - pre;
        }
        uint32_t t1, t2;
        const uint32_t e1 = warp_excl_sum(cnt, t1);
        const uint32_t e2 = warp_excl_sum(pre, t2);
        if (lane == 31) { s_scan[0][warp] = t1; s_scan[1][warp] = t2; }
        __syncthreads();
        uint32_t p1 = 0, p2 = 0;
        for (uint32_t w = 0; w < warp; ++w) { p1 += s_scan[0][w]; p2 += s_scan[1][w]; }
        s_tcum[tid] = p1 + e1;
        s_gcum[tid] = p2 + e2;
        if (tid == 255) { s_tcum[256] = p1 + e1 + cnt; s_gcum[256] = p2 + e2 + pre; }
    }
    if (tid == 0) s_wp[WTL_THREADS].x = 0;
    // symbols -> paths, original order (32 consecutive symbols per thread: two 16-byte loads)
    {
        const uint8_t *src = sym + base + (uint64_t)tid * WTL_EPT;
        const bool vec = ((reinterpret_cast<uintptr_t>(sym) & 15) == 0) && (tid * WTL_EPT + WTL_EPT <= nv);
        if (vec) {
            const uint4 *q = reinterpret_cast<const uint4 *>(src);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint4 x = q[h];
                const uint32_t w4[4] = {x.x, x.y, x.z, x.w};
                uint32_t o4[4];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    o4[j] = (uint32_t)s_path[w4[j] & 0xFF] | ((uint32_t)s_path[(w4[j] >> 8) & 0xFF] << 8) |
                            ((uint32_t)s_path[(w4[j] >> 16) & 0xFF] << 16) | ((uint32_t)s_path[w4[j] >> 24] << 24);
                reinterpret_cast<uint4 *>(s_a + tid * WTL_EPT)[h] = make_uint4(o4[0], o4[1], o4[2], o4[3]);
            }
        } else {
            for (uint32_t k = 0; k < WTL_EPT; ++k) {
                const uint32_t i = tid * WTL_EPT + k;
                s_a[i] = (i < nv) ? s_path[src[k]] : (uint8_t)0xFF;
            }
        }
    }
    __syncthreads();

    uint8_t *cur = s_a, *nxt = s_b;
    const uint32_t lt = lanemask_lt(), lanebit = 1u << lane;
    for (uint32_t l = 0; l < levels; ++l) {
        const uint32_t shift = 7u - l;
        // ---- A: the words of bits of this warp's 32 rows (lane 0 files each), ones before every row
        const uint8_t *wrow = cur + warp * 1024u + lane;
        uint2 *wp_row = s_wp + warp * 32u;
#pragma unroll 8
        for (uint32_t r = 0; r < 32; ++r) {
            const uint32_t pth = wrow[r * 32u];
            const uint32_t word = __ballot_sync(0xffffffffu, (pth >> shift) & 1u);
            if (lane == 0) wp_row[r].x = word;
        }
        __syncwarp();
        {
            const uint32_t myword = s_wp[tid].x;
            uint32_t wt;
            const uint32_t ex = warp_excl_sum(__popc(myword), wt);
            if (lane == 31) s_scan[0][warp] = wt;
            __syncthreads();
            uint32_t p = 0, tot = 0;
            for (uint32_t q = 0; q < WTL_THREADS / 32; ++q) { if (q < warp) p += s_scan[0][q]; tot += s_scan[0][q]; }
            s_wp[tid].y = p + ex;
            if (tid == 0) s_wp[WTL_THREADS].y = tot;
        }
        __syncthreads();
        // ---- B: every internal node's run of bits into the level (warps take nodes round-robin)
        {
            const uint32_t nnodes = tab->lvl_nodes[l];
            uint32_t *words = lv.w[l];
            for (uint32_t k = warp; k < nnodes; k += WTL_THREADS / 32) {
                const uint32_t lo = tab->lvl_lo[l][k], hi = (uint32_t)tab->lvl_hi1[l][k] + 1;
                const uint32_t x0 = tab->path_of_code[lo], x1 = tab->path_of_code[hi];
                const uint32_t s0 = s_tcum[x0], r = s_tcum[x1] - s0;
                if (r == 0) continue;
                const uint32_t D = (tab->node_start[l][lo] & NODE_START_MASK) + (s_gcum[x1] - s_gcum[x0]);
                const uint32_t q0 = D >> 5, q1 = (D + r - 1) >> 5;
                for (uint32_t q = q0 + lane; q <= q1; q += 32) {
                    const uint32_t lo_bit = max(q << 5, D), hi_bit = min((q << 5) + 32u, D + r);
                    const uint32_t nb = hi_bit - lo_bit;
                    const uint32_t i0 = s0 + (lo_bit - D);
                    const uint32_t wi = i0 >> 5, sh = i0 & 31u;
                    const uint64_t x = (uint64_t)s_wp[wi].x | ((uint64_t)s_wp[wi + 1].x << 32);
                    uint32_t v = (uint32_t)(x >> sh);
                    if (nb < 32) v &= (1u << nb) - 1u;
                    const uint32_t out = v << (lo_bit - (q << 5));
                    uint32_t *dst = words + (size_t)(q / 7u) * 8u + 1u + (q % 7u);
                    if (nb == 32) *dst = out;
                    else if (out) atomicOr(dst, out);
                }
            }
        }
        if (l + 1 == levels) break;
        // ---- C: stable split of every run by its bit -> order by the top l + 1 path bits
        if (tid < (1u << l)) {
            const uint32_t x_lo = tid << (shift + 1u);
            const uint32_t S = s_tcum[x_lo], M = s_tcum[x_lo + (1u << shift)];
            const uint2 wp = s_wp[S >> 5];
            const uint32_t ps = wp.y + __popc(wp.x & ((1u << (S & 31u)) - 1u));
            s_ent[tid] = (M - ps) | (ps << 16);
        }
        __syncthreads();
        {
            uint8_t *wout = nxt;
            const uint32_t i0 = warp * 1024u + lane;
#pragma unroll 8
            for (uint32_t r = 0; r < 32; ++r) {
                const uint32_t pth = wrow[r * 32u];
                const uint2 wp = wp_row[r];                               // the row's word and the ones before it: a broadcast
                const uint32_t e = s_ent[pth >> (shift + 1u)];
                const uint32_t ob = wp.y + __popc(wp.x & lt);             // ones before this element in the tile order
                const uint32_t dst = (wp.x & lanebit) ? (e & 0xFFFFu) + ob : (i0 + r * 32u) + (e >> 16) - ob;
                wout[dst] = (uint8_t)pth;
            }
        }
        __syncthreads();
        uint8_t *t = cur; cur = nxt; nxt = t;
    }
}

// Headers for a level whose payload bits are already in place: per rank block, ones before it
// inside this CTA's 256-block tile; tile totals to agg.
constexpr int WTC_BLOCKS_PER_CTA = 256;

// The directories of ALL levels in three launches (count, scan, fix) instead of three per level: the tiles of rank
// blocks of every level are numbered consecutively (tile0[l] = first tile of level l) in agg / carry.  A bit vector
// packed by dir_store_tile is a one-level description with tiles of WTP_BLOCKS_PER_CTA blocks.
struct DirLevels {
    RankBlock *blocks[HKCSA_MAX_LEVELS];
    uint64_t *super[HKCSA_MAX_LEVELS];
    uint32_t *select[HKCSA_MAX_LEVELS];
    uint64_t nblocks[HKCSA_MAX_LEVELS];
    uint32_t tile0[HKCSA_MAX_LEVELS + 1];
    uint32_t levels;
};

__device__ __forceinline__ uint32_t dir_level_of_tile(const DirLevels &D, uint32_t tile)
{
    uint32_t l = 0;
    while (l + 1 < D.levels && tile >= D.tile0[l + 1]) ++l;
    return l;
}

__global__ void __launch_bounds__(WTC_BLOCKS_PER_CTA)
wt_count_all_kernel(DirLevels D, uint32_t *__restrict__ agg)
{
    const uint32_t tid = threadIdx.x;
    const uint32_t l = dir_level_of_tile(D, blockIdx.x);
    RankBlock *blocks = D.blocks[l];
    const uint64_t nblocks = D.nblocks[l];
    const uint64_t g = (uint64_t)(blockIdx.x - D.tile0[l]) * WTC_BLOCKS_PER_CTA + tid;
    uint32_t cnt = 0;
    if (g < nblocks) {
        const RankBlock b = load_block(blocks + g);
        cnt = block_rank(b, HKCSA_BLOCK_BITS);
    }
    uint32_t total;
    const uint32_t ex = block_excl_scan(cnt, 0u, Plus(), total);
    if (g < nblocks) reinterpret_cast<uint32_t *>(blocks + g)[0] = ex;
    if (tid == 0) agg[blockIdx.x] = total;
}

// CTA l: exclusive scan of level l's tile totals -> carry (same numbering); ones of the level -> ones_out[l]
__global__ void __launch_bounds__(1024)
wt_dir_scan_all_kernel(DirLevels D, const uint32_t *__restrict__ agg, uint64_t *__restrict__ carry,
                       uint64_t *__restrict__ ones_out)
{
    const uint32_t l = blockIdx.x, t0 = D.tile0[l];
    const uint64_t ones = block_excl_scan_carried(D.tile0[l + 1] - t0, (uint64_t)0, Plus(),
                                                  [&](uint32_t t) { return (uint64_t)agg[t0 + t]; },
                                                  [&](uint32_t t, uint64_t p) { carry[t0 + t] = p; });
    if (threadIdx.x == 0) ones_out[l] = ones;
}

// one thread per rank block, CTAs of 256 blocks.  With TILE = 256 CTA c is tile c, which places it in its level; a
// description with smaller tiles has one level.
template <uint32_t TILE>
__global__ void __launch_bounds__(WTC_BLOCKS_PER_CTA)
wt_dir_fix_all_kernel(DirLevels D, const uint64_t *__restrict__ carry)
{
    const uint32_t l = dir_level_of_tile(D, blockIdx.x);
    const uint64_t g = (uint64_t)(blockIdx.x - D.tile0[l]) * WTC_BLOCKS_PER_CTA + threadIdx.x;
    if (g >= D.nblocks[l]) return;
    dir_finish_block<TILE>(load_block(D.blocks[l] + g), g, D.blocks[l], carry + D.tile0[l], D.super[l], D.select[l]);
}

// node_ones[l][code] = rank1(level l, start of code's node)
__global__ void wt_node_ones_kernel(WtDev wt, WtTables *tab)
{
    const uint32_t l = blockIdx.x, c = threadIdx.x;
    if (l >= wt.levels || c >= wt.sigma) return;
    if (tab->depth[c] <= l) { tab->node_ones[l][c] = 0; return; }
    const uint32_t start = tab->node_start[l][c] & NODE_START_MASK;
    tab->node_ones[l][c] = (uint32_t)bv_rank(wt.level[l], start);
}

// ---------------------------------------------------------------- bit-vector queries
__global__ void bv_rank_kernel(BitVec v, const uint64_t *__restrict__ pos, uint64_t m, uint64_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const uint64_t i = min(pos[q], v.len);
    out[q] = bv_rank(v, i);
}

__device__ __forceinline__ uint64_t bv_block_abs(const BitVec &v, uint64_t g)
{
    const uint32_t hdr = reinterpret_cast<const uint32_t *>(v.blocks + g)[0];
    return v.super[g / HKCSA_SUPER_BLOCKS] + hdr;
}

// select(k): smallest p in [0, len] with rank(p) >= k  (csa/wavelet_tree.py:17-25)
__global__ void bv_select_kernel(BitVec v, const uint32_t *__restrict__ samples, uint64_t ones,
                                 const uint64_t *__restrict__ ks, uint64_t m, uint64_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const uint64_t k = ks[q];
    if (k == 0) { out[q] = 0; return; }
    if (k > ones) { out[q] = v.len; return; }
    const uint64_t t = (k - 1) / HKCSA_SELECT_SAMPLE;
    uint64_t lo = samples[t] / HKCSA_BLOCK_BITS;                    // block holding one number 1+t*S
    const uint64_t last = v.len / HKCSA_BLOCK_BITS;
    uint64_t hi = ((t + 1) * HKCSA_SELECT_SAMPLE + 1 <= ones) ? samples[t + 1] / HKCSA_BLOCK_BITS : last;
    // last block g in [lo, hi] with abs_before(g) < k
    while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) / 2;
        if (bv_block_abs(v, mid) < k) lo = mid; else hi = mid - 1;
    }
    const RankBlock b = load_block(v.blocks + lo);
    const uint32_t r = (uint32_t)(k - bv_block_abs(v, lo));
    out[q] = lo * HKCSA_BLOCK_BITS + block_select(b, r) + 1;
}

__global__ void bv_unpack_kernel(BitVec v, uint64_t begin, uint64_t count, uint8_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    const uint64_t i = begin + q;
    const uint64_t g = i / HKCSA_BLOCK_BITS;
    const RankBlock b = load_block(v.blocks + g);
    out[q] = (uint8_t)block_bit(b, (uint32_t)(i - g * HKCSA_BLOCK_BITS));
}

__global__ void bv_rank_range_kernel(BitVec v, uint64_t begin, uint64_t count, uint32_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    out[q] = (uint32_t)bv_rank(v, begin + q);
}

// ---------------------------------------------------------------- symbol-level queries
__global__ void __launch_bounds__(256)
wt_rank_kernel(WtDev wt, const uint8_t *__restrict__ sym, const uint64_t *__restrict__ pos, uint64_t m,
               uint64_t *__restrict__ out)
{
    __shared__ WtSmem s;
    wt_smem_load(s, wt);
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const uint32_t code = s.code_of_sym[sym[q]];
    if (code == 0xFFFFu) { out[q] = 0; return; }            // "character not in occ" -> 0
    const uint64_t i = min(pos[q], wt.n);                    // index clamp of enhanced_fm_index.py:37-38
    if (wt.sigma == 1) { out[q] = i; return; }
    out[q] = wt_rank_code(s, wt, code, (uint32_t)i);
}

__global__ void __launch_bounds__(256)
wt_access_kernel(WtDev wt, const uint64_t *__restrict__ pos, uint64_t m, uint8_t *__restrict__ out)
{
    __shared__ WtSmem s;
    wt_smem_load(s, wt);
    __syncthreads();
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    uint32_t occ;
    const uint32_t code = wt_access_rank(s, wt, (uint32_t)pos[q], occ);
    out[q] = s.sym_of_code[code];
}

}  // namespace hkcsa

// ------------------------------------------------------------------ host side
using namespace hkcsa;

// Directory scratch of `levels` levels of at most n bits, in tiles of `tile_blocks` rank blocks: tile totals and
// carries (numbered as in DirLevels) and the ones of every level.
struct DirScratch {
    uint32_t *agg;
    uint64_t *carry;
    uint64_t *ones;
};
static DirScratch carve_dir_scratch(Carver &c, uint64_t n, uint32_t levels, uint32_t tile_blocks)
{
    const uint64_t tiles = levels * (rank_blocks_for(n) / tile_blocks + 2);
    DirScratch d;
    d.agg = c.take<uint32_t>(tiles);
    d.carry = c.take<uint64_t>(tiles);
    d.ones = c.take<uint64_t>(HKCSA_MAX_LEVELS);
    return d;
}

// scratch of hkcsa_wt_build: per-symbol tile counts, then the directories of all levels
static size_t wt_scratch_for(uint64_t n, uint32_t sigma)
{
    Carver c(nullptr);
    const uint64_t wtiles = (n + WTL_TILE - 1) / WTL_TILE;
    c.take<uint32_t>((uint64_t)(sigma ? sigma : 1) * (wtiles + 1));
    carve_dir_scratch(c, n, HKCSA_MAX_LEVELS, WTC_BLOCKS_PER_CTA);
    return c.total();
}

// The blob of a plan: the node tables, then per level of level_len[l] bits (0 past the tree) its rank blocks,
// superblocks and select samples, each 256-byte aligned.
static void wt_layout_blob(hkcsa_wt_plan *p)
{
    uint64_t off = 0;
    p->off_tables = off;
    off = align_up(off + sizeof(WtTables), 256);
    for (uint32_t l = 0; l < HKCSA_MAX_LEVELS; ++l) {
        const uint64_t bits = p->level_len[l];
        p->off_blocks[l] = off;
        off = align_up(off + rank_blocks_for(bits) * sizeof(RankBlock), 256);
        p->off_super[l] = off;
        off = align_up(off + super_for(bits) * sizeof(uint64_t), 256);
        p->off_select[l] = off;
        off = align_up(off + select_samples_for(bits) * sizeof(uint32_t), 256);
    }
    p->blob_bytes = off;
}

// the one-level description of a bit vector of nbits bits packed by dir_store_tile
static DirLevels packed_dir(RankBlock *blocks, uint64_t *super, uint32_t *select, uint64_t nbits)
{
    DirLevels D;
    memset(&D, 0, sizeof(D));
    D.levels = 1;
    D.blocks[0] = blocks;
    D.super[0] = super;
    D.select[0] = select;
    D.nblocks[0] = rank_blocks_for(nbits);
    D.tile0[1] = (uint32_t)((D.nblocks[0] + WTP_BLOCKS_PER_CTA - 1) / WTP_BLOCKS_PER_CTA);
    return D;
}

extern "C" int hkcsa_wt_plan_from_hist(const uint64_t h_hist[256], hkcsa_wt_plan *p)
{
    HK_REQUIRE(h_hist && p, HKCSA_EINVAL, "null pointer");
    memset(p, 0, sizeof(*p));
    uint64_t n = 0;
    uint32_t sigma = 0;
    for (int ch = 0; ch < 256; ++ch) {
        p->code_of_sym[ch] = 0xFFFF;
        if (h_hist[ch]) {
            p->code_of_sym[ch] = (uint16_t)sigma;
            p->sym_of_code[sigma] = (uint8_t)ch;
            p->cnt[sigma] = h_hist[ch];
            p->C[sigma] = n;
            n += h_hist[ch];
            ++sigma;
        }
    }
    p->C[sigma] = n;
    p->n = n;
    p->sigma = sigma;
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    memset(p->node_id, 0xFF, sizeof(p->node_id));
    // breadth-first over the alphabet-halving tree
    struct Node { uint32_t lo, hi; };
    Node cur[256], nxt[256];
    uint32_t ncur = 0;
    if (sigma >= 2) cur[ncur++] = {0, sigma};
    uint32_t level = 0;
    while (ncur) {
        HK_REQUIRE(level < HKCSA_MAX_LEVELS, HKCSA_EINVAL, "internal: tree deeper than 8 levels");
        uint64_t start = 0;
        uint32_t nn = 0;
        for (uint32_t k = 0; k < ncur; ++k) {
            const uint32_t lo = cur[k].lo, hi = cur[k].hi, mid = lo + (hi - lo) / 2;
            uint64_t sz = 0;
            for (uint32_t c = lo; c < hi; ++c) {
                p->node_start[level][c] = (uint32_t)start;
                p->node_bit[level][c] = (c >= mid);
                p->node_id[level][c] = (uint8_t)k;
                p->depth[c]++;
                sz += p->cnt[c];
            }
            start += sz;
            if (mid - lo >= 2) nxt[nn++] = {lo, mid};
            if (hi - mid >= 2) nxt[nn++] = {mid, hi};
        }
        p->level_len[level] = start;
        p->level_nodes[level] = ncur;
        memcpy(cur, nxt, nn * sizeof(Node));
        ncur = nn;
        ++level;
    }
    p->levels = level;
    wt_layout_blob(p);
    p->scratch_bytes = wt_scratch_for(n, sigma);
    return HKCSA_OK;
}

// the largest blob / scratch a plan over n symbols can ask for (256 symbols, 8 levels): what a caller allocates
// before the byte histogram is known (hkcsa_index_build)
extern "C" size_t hkcsa_wt_blob_bound(uint64_t n)
{
    hkcsa_wt_plan p;
    for (uint32_t l = 0; l < HKCSA_MAX_LEVELS; ++l) p.level_len[l] = n;
    wt_layout_blob(&p);
    return p.blob_bytes;
}
extern "C" size_t hkcsa_wt_scratch_bound(uint64_t n) { return wt_scratch_for(n, 256); }

// Sampled suffix array with the suffix array streamed ONCE: `ssa_mark_pack_kernel` packs the mark bit-vector (bit j =
// SA[j] % rate == 0) into rank blocks -- a thread takes four consecutive rows per step (one 16-byte load for 32-bit
// ids), the flag nibbles of eight lanes are OR-ed into the 32-bit word of their rows with three shuffles --, the
// directory scan turns the tile totals into carries, and `ssa_fix_sample_kernel` finishes the directory and writes
// the samples SA[j] / rate of the marked rows in row order: the thread of a rank block knows the marks before it and
// reads only the marked entries again (one in `rate`).  (A single kernel with a decoupled look-back over one counter
// per 14336-row tile was measured first: its chain of inclusive prefixes advances 32 tiles per L2 round trip, 218 hops
// for C2 = 0.25 ms whatever the bandwidth.)
namespace hkcsa {
constexpr int SSA_STEPS = WTP_SYMS / (WTP_THREADS * 4);      // 14 steps of 1024 rows
static_assert(WTP_SYMS % (WTP_THREADS * 4) == 0, "tile shape");
constexpr int SSA_WORDS = WTP_SYMS / 32;                     // 448 words = 64 blocks x 7

template <typename IdT>
__device__ __forceinline__ void ssa_load4_fast(const IdT *__restrict__ p, IdT v[4])
{
    if constexpr (sizeof(IdT) == 4) {
        const uint4 q = *reinterpret_cast<const uint4 *>(p);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
        const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(p);
        const ulonglong2 b = *reinterpret_cast<const ulonglong2 *>(p + 2);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
}

template <typename IdT>
__device__ __forceinline__ void ssa_load4(const IdT *__restrict__ sa, uint64_t n, uint64_t r0, bool aligned16, IdT v[4])
{
    if (r0 + 4 <= n && aligned16) {
        if constexpr (sizeof(IdT) == 4) {
            const uint4 q = *reinterpret_cast<const uint4 *>(sa + r0);
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
            const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(sa + r0);
            const ulonglong2 b = *reinterpret_cast<const ulonglong2 *>(sa + r0 + 2);
            v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = (r0 + e < n) ? sa[r0 + e] : (IdT)1;      // 1 % rate != 0 unless rate == 1: masked below
    }
}

// the flags of the tile's rows: every thread's four flags per step (returned), the words of 32 rows into s_words
template <typename IdT, bool POW2, bool FAST>
__device__ __forceinline__ uint64_t ssa_flag_steps(const IdT *__restrict__ sa, uint64_t n, uint64_t row_base, uint32_t rate,
                                                   IdT mask, bool aligned16, uint32_t *s_words)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t nib_shift = 4u * (lane & 7u);
    uint32_t *my_word = &s_words[warp * 4 + (lane >> 3)];
    const IdT *p = sa + row_base + tid * 4u;
    uint64_t nibs = 0;
#pragma unroll
    for (int it = 0; it < SSA_STEPS; ++it) {
        IdT v[4];
        if (FAST) ssa_load4_fast<IdT>(p + it * (WTP_THREADS * 4), v);
        else ssa_load4<IdT>(sa, n, row_base + (uint64_t)it * (WTP_THREADS * 4) + tid * 4u, aligned16, v);
        uint32_t nib = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const bool hit = POW2 ? ((v[e] & mask) == 0) : (v[e] % rate == 0);
            const bool f = hit && (FAST || row_base + (uint64_t)it * (WTP_THREADS * 4) + tid * 4u + e < n);
            nib |= (f ? 1u : 0u) << e;
        }
        nibs |= (uint64_t)nib << (4 * it);
        uint32_t x = nib << nib_shift;
        x |= __shfl_xor_sync(0xffffffffu, x, 1);
        x |= __shfl_xor_sync(0xffffffffu, x, 2);
        x |= __shfl_xor_sync(0xffffffffu, x, 4);
        if ((lane & 7u) == 0) my_word[it * (WTP_THREADS / 8)] = x;
    }
    return nibs;
}

// POW2: the rate is a power of two -- a mask and a shift per entry instead of a division (a run-time test inside the
// loop made the compiler evaluate both forms for every entry: 37 instructions per row)
template <typename IdT, bool POW2>
__global__ void __launch_bounds__(WTP_THREADS)
ssa_mark_pack_kernel(const IdT *__restrict__ sa, uint64_t n, uint32_t rate, RankBlock *__restrict__ blocks,
                     uint64_t nblocks, uint32_t *__restrict__ agg)
{
    __shared__ uint32_t s_words[SSA_WORDS];
    const uint32_t tid = threadIdx.x;
    const uint32_t tile = blockIdx.x;
    const uint64_t row_base = (uint64_t)tile * WTP_SYMS;
    const IdT mask = (IdT)(rate - 1u);
    const bool aligned16 = (reinterpret_cast<uintptr_t>(sa) & 15) == 0;
    const bool fast = aligned16 && row_base + WTP_SYMS <= n;     // every tile but the last: no bounds checks
    if (fast) ssa_flag_steps<IdT, POW2, true>(sa, n, row_base, rate, mask, aligned16, s_words);
    else ssa_flag_steps<IdT, POW2, false>(sa, n, row_base, rate, mask, aligned16, s_words);
    __syncthreads();
    dir_store_tile(s_words, blocks, nblocks, tile, agg);
}

// The directory of the mark vector (dir_finish_block), and the samples: the thread of a rank block knows the marks
// before it and walks the block's set bits in row order: samples[marks before + k] = SA[row] / rate.  Only the marked
// entries are read again -- one in `rate`, 7 per block at rate 32 -- so the suffix array is streamed once.
template <typename IdT, bool POW2>
__global__ void __launch_bounds__(256)
ssa_fix_sample_kernel(RankBlock *__restrict__ blocks, uint64_t nblocks, const uint64_t *__restrict__ carry,
                      uint64_t *__restrict__ super, uint32_t *__restrict__ select_samples, const IdT *__restrict__ sa,
                      uint32_t rate, uint32_t *__restrict__ samples)
{
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nblocks) return;
    const RankBlock b = load_block(blocks + g);
    const BlockOnes ones = dir_finish_block<WTP_BLOCKS_PER_CTA>(b, g, blocks, carry, super, select_samples);
    if (ones.in == 0) return;
    const int sh = __ffs(rate) - 1;
    const IdT *row0 = sa + g * HKCSA_BLOCK_BITS;
    uint32_t *out = samples + ones.before;
    uint32_t k = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint64_t x = q ? b.w[q] : (b.w[0] >> 32);          // payload bit j of the block = bit 32 + j of the 256
        const int base = q ? 64 * q - 32 : 0;
        while (x) {
            const int bit = __ffsll((long long)x) - 1;
            x &= x - 1;
            const IdT v = row0[base + bit];
            out[k++] = POW2 ? (uint32_t)(v >> sh) : (uint32_t)(v / rate);
        }
    }
}
}  // namespace hkcsa

// the sampled SA's scratch: the directory of the mark vector and its select samples (the blob keeps none)
struct SsaScratch {
    DirScratch dir;
    uint32_t *select;
};
static SsaScratch carve_ssa_scratch(Carver &c, uint64_t n)
{
    SsaScratch s;
    s.dir = carve_dir_scratch(c, n, 1, WTP_BLOCKS_PER_CTA);
    s.select = c.take<uint32_t>(select_samples_for(n));
    return s;
}

extern "C" int hkcsa_ssa_plan_make(uint64_t n, uint32_t rate, hkcsa_ssa_plan *p)
{
    HK_REQUIRE(p && rate >= 1, HKCSA_EINVAL, "bad argument");
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    memset(p, 0, sizeof(*p));
    p->n = n;
    p->rate = rate;
    p->n_samples = (n + rate - 1) / rate;
    uint64_t off = 0;
    p->off_blocks = off;
    off = align_up(off + rank_blocks_for(n) * sizeof(RankBlock), 256);
    p->off_super = off;
    off = align_up(off + super_for(n) * sizeof(uint64_t), 256);
    p->off_samples = off;
    off = align_up(off + (p->n_samples + 1) * sizeof(uint32_t), 256);
    p->blob_bytes = off;
    Carver c(nullptr);
    carve_ssa_scratch(c, n);
    p->scratch_bytes = c.total();
    return HKCSA_OK;
}

extern "C" int hkcsa_ssa_plan_make_slice(uint64_t m, uint32_t rate, uint64_t n_marks, hkcsa_ssa_plan *p)
{
    int rc = hkcsa_ssa_plan_make(m, rate, p);
    if (rc != HKCSA_OK) return rc;
    HK_REQUIRE(n_marks <= m, HKCSA_EINVAL, "more marks than rows");
    p->n_samples = n_marks;
    p->off_samples = p->off_super + align_up(super_for(m) * sizeof(uint64_t), 256);
    p->blob_bytes = p->off_samples + align_up((n_marks + 1) * sizeof(uint32_t), 256);
    return HKCSA_OK;
}

// mark vector, directory and samples in one pass over d_sa: ids read once (+ the marked ones again from cache)
template <typename IdT>
static int ssa_build_t(const IdT *d_sa, const hkcsa_ssa_plan *p, void *d_blob, void *d_scratch, size_t scratch_bytes,
                       void *stream)
{
    HK_REQUIRE(p && d_blob && d_scratch && (d_sa || p->n == 0), HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(p->scratch_bytes <= scratch_bytes, HKCSA_ESCRATCH, "sampled-SA scratch too small");
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_blob) & 31) == 0, HKCSA_EINVAL, "blob must be 32-byte aligned");
    cudaStream_t st = as_stream(stream);
    const uint64_t n = p->n;
    const uint32_t rate = p->rate;
    if (n == 0) return HKCSA_OK;
    Carver c(d_scratch);
    const SsaScratch s = carve_ssa_scratch(c, n);
    const DirScratch &dir = s.dir;
    uint8_t *blob = static_cast<uint8_t *>(d_blob);
    const DirLevels D = packed_dir(reinterpret_cast<RankBlock *>(blob + p->off_blocks),
                                   reinterpret_cast<uint64_t *>(blob + p->off_super), s.select, n);
    RankBlock *blocks = D.blocks[0];
    const uint64_t nblocks = D.nblocks[0];
    uint32_t *samples = reinterpret_cast<uint32_t *>(blob + p->off_samples);
    prof::Scope ps(st, prof::SSA_BUILD, n * sizeof(IdT) + n / 7 + (n / rate) * (4 + sizeof(IdT)));
    const bool pow2 = (rate & (rate - 1u)) == 0;
    if (pow2) ssa_mark_pack_kernel<IdT, true><<<D.tile0[1], WTP_THREADS, 0, st>>>(d_sa, n, rate, blocks, nblocks, dir.agg);
    else ssa_mark_pack_kernel<IdT, false><<<D.tile0[1], WTP_THREADS, 0, st>>>(d_sa, n, rate, blocks, nblocks, dir.agg);
    HK_LAUNCH_CHECK();
    wt_dir_scan_all_kernel<<<1, 1024, 0, st>>>(D, dir.agg, dir.carry, dir.ones);
    HK_LAUNCH_CHECK();
    const uint32_t grid = (uint32_t)((nblocks + 255) / 256);
    if (pow2) ssa_fix_sample_kernel<IdT, true><<<grid, 256, 0, st>>>(blocks, nblocks, dir.carry, D.super[0], s.select, d_sa, rate, samples);
    else ssa_fix_sample_kernel<IdT, false><<<grid, 256, 0, st>>>(blocks, nblocks, dir.carry, D.super[0], s.select, d_sa, rate, samples);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_ssa_build(const uint32_t *d_sa, const hkcsa_ssa_plan *p, void *d_blob, void *d_scratch,
                               size_t scratch_bytes, void *stream)
{
    return ssa_build_t<uint32_t>(d_sa, p, d_blob, d_scratch, scratch_bytes, stream);
}

// suffix ids as uint64 (slices of a text beyond 4 GB); samples stay uint32 (id / rate must fit)
extern "C" int hkcsa_ssa_build64(const uint64_t *d_sa, const hkcsa_ssa_plan *p, void *d_blob, void *d_scratch,
                                 size_t scratch_bytes, void *stream)
{
    return ssa_build_t<uint64_t>(d_sa, p, d_blob, d_scratch, scratch_bytes, stream);
}

// host-side node tables of a plan -> the blob's table region
static int wt_write_tables(const hkcsa_wt_plan *p, uint8_t *blob, cudaStream_t st)
{
    static thread_local WtTables T;   // staged from pageable memory (a few KB, once per build)
    memset(&T, 0, sizeof(T));
    memcpy(T.code_of_sym, p->code_of_sym, sizeof(T.code_of_sym));
    memcpy(T.sym_of_code, p->sym_of_code, sizeof(T.sym_of_code));
    memcpy(T.depth, p->depth, sizeof(T.depth));
    for (uint32_t c = 0; c <= p->sigma && c < 260; ++c) T.C[c] = (uint32_t)p->C[c];
    for (uint32_t l = 0; l < p->levels; ++l) {
        for (uint32_t c = 0; c < p->sigma; ++c) {
            T.node_start[l][c] = p->node_start[l][c] | (p->node_bit[l][c] ? NODE_BIT_FLAG : 0u);
        }
        // node extents: per code and per node
        uint32_t lo_of[256], hi_of[256];
        for (uint32_t k = 0; k < 256; ++k) { lo_of[k] = 0xFFFFFFFFu; hi_of[k] = 0; }
        for (uint32_t c = 0; c < p->sigma; ++c) {
            const uint8_t id = p->node_id[l][c];
            if (id == 0xFF) continue;
            if (lo_of[id] == 0xFFFFFFFFu) lo_of[id] = c;
            hi_of[id] = c;
        }
        for (uint32_t c = 0; c < p->sigma; ++c) {
            const uint8_t id = p->node_id[l][c];
            if (id == 0xFF) continue;
            T.node_lo[l][c] = (uint8_t)lo_of[id];
            T.node_hi1[l][c] = (uint8_t)hi_of[id];
        }
        T.lvl_nodes[l] = p->level_nodes[l];
        for (uint32_t k = 0; k < p->level_nodes[l] && k < 128; ++k) {
            T.lvl_lo[l][k] = (uint8_t)lo_of[k];
            T.lvl_hi1[l][k] = (uint8_t)hi_of[k];
        }
    }
    for (int ch = 0; ch < 256; ++ch) T.code8_of_sym[ch] = (p->code_of_sym[ch] == 0xFFFF) ? 0 : (uint8_t)p->code_of_sym[ch];
    memset(T.code_of_path, 0xFF, sizeof(T.code_of_path));
    for (uint32_t c = 0; c < p->sigma; ++c) {
        uint32_t path = 0;
        for (uint32_t l = 0; l < p->depth[c]; ++l) path |= (uint32_t)(p->node_bit[l][c] ? 1u : 0u) << (7 - l);
        T.path_of_code[c] = (uint16_t)path;
        T.code_of_path[path] = (uint16_t)c;
        T.path_of_sym[p->sym_of_code[c]] = (uint8_t)path;
    }
    T.path_of_code[p->sigma] = 256;
    WtTables *d_tab = reinterpret_cast<WtTables *>(blob + p->off_tables);
    // pageable source: the call returns once T has been copied to the driver's staging buffer (no wait for the
    // stream), so T may be reused by the next call on this thread and the host goes on enqueueing the build
    HK_CUDA(cudaMemcpyAsync(d_tab, &T, sizeof(T), cudaMemcpyHostToDevice, st));
    return HKCSA_OK;
}

// block headers, superblocks and select samples of every level from the payload bits in place; node_ones; syncs
// once to read the ones per level (h_ones_out[levels])
static int wt_build_dirs(const hkcsa_wt_plan *p, void *d_blob, const DirScratch &dir, uint64_t *h_ones_out,
                         cudaStream_t st)
{
    uint8_t *blob = static_cast<uint8_t *>(d_blob);
    WtTables *d_tab = reinterpret_cast<WtTables *>(blob + p->off_tables);
    DirLevels D;
    memset(&D, 0, sizeof(D));
    D.levels = p->levels;
    uint64_t all_blocks = 0;
    for (uint32_t l = 0; l < p->levels; ++l) {
        D.blocks[l] = reinterpret_cast<RankBlock *>(blob + p->off_blocks[l]);
        D.super[l] = reinterpret_cast<uint64_t *>(blob + p->off_super[l]);
        D.select[l] = reinterpret_cast<uint32_t *>(blob + p->off_select[l]);
        D.nblocks[l] = rank_blocks_for(p->level_len[l]);
        D.tile0[l + 1] = D.tile0[l] + (uint32_t)((D.nblocks[l] + WTC_BLOCKS_PER_CTA - 1) / WTC_BLOCKS_PER_CTA);
        all_blocks += D.nblocks[l];
    }
    if (D.tile0[p->levels]) {
        prof::Scope ps(st, prof::WT_DIR, all_blocks * 72);
        wt_count_all_kernel<<<D.tile0[p->levels], WTC_BLOCKS_PER_CTA, 0, st>>>(D, dir.agg);
        HK_LAUNCH_CHECK();
        wt_dir_scan_all_kernel<<<p->levels, 1024, 0, st>>>(D, dir.agg, dir.carry, dir.ones);
        HK_LAUNCH_CHECK();
        wt_dir_fix_all_kernel<WTC_BLOCKS_PER_CTA><<<D.tile0[p->levels], WTC_BLOCKS_PER_CTA, 0, st>>>(D, dir.carry);
        HK_LAUNCH_CHECK();
    }
    WtDev wt = make_wt_dev(d_blob, p);
    wt_node_ones_kernel<<<p->levels, 256, 0, st>>>(wt, d_tab);
    HK_LAUNCH_CHECK();
    uint64_t *h_ones = reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(pinned_page()) + 3072);
    HK_CUDA(cudaMemcpyAsync(h_ones, dir.ones, p->levels * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    for (uint32_t l = 0; l < p->levels; ++l) h_ones_out[l] = h_ones[l];
    return HKCSA_OK;
}

extern "C" int hkcsa_wt_build(const uint8_t *d_sym, hkcsa_wt_plan *p, void *d_blob, void *d_scratch,
                              size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(p && d_blob, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(p->scratch_bytes <= scratch_bytes, HKCSA_ESCRATCH, "wavelet scratch too small");
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_blob) & 31) == 0, HKCSA_EINVAL, "blob must be 32-byte aligned");
    cudaStream_t st = as_stream(stream);
    const uint64_t n = p->n;
    uint8_t *blob = static_cast<uint8_t *>(d_blob);
    int rc = wt_write_tables(p, blob, st);
    if (rc != HKCSA_OK) return rc;
    WtTables *d_tab = reinterpret_cast<WtTables *>(blob + p->off_tables);
    if (p->levels == 0 || n == 0) return HKCSA_OK;
    HK_REQUIRE(d_sym && d_scratch, HKCSA_EINVAL, "null pointer");

    Carver c(d_scratch);
    const uint32_t wtiles = (uint32_t)((n + WTL_TILE - 1) / WTL_TILE);
    uint32_t *d_gcnt = c.take<uint32_t>((uint64_t)p->sigma * (wtiles + 1));
    const DirScratch dir = carve_dir_scratch(c, n, HKCSA_MAX_LEVELS, WTC_BLOCKS_PER_CTA);

    // payload bits are OR-ed in: the level regions must start from zero
    HK_CUDA(cudaMemsetAsync(blob + p->off_blocks[0], 0, p->blob_bytes - p->off_blocks[0], st));
    LevelWords lw;
    for (uint32_t l = 0; l < HKCSA_MAX_LEVELS; ++l) lw.w[l] = reinterpret_cast<uint32_t *>(blob + p->off_blocks[l]);
    {
        prof::Scope ps(st, prof::WT_LEVELS, n + (uint64_t)p->levels * (n / 8));
        wt_tile_hist_kernel<<<wtiles, WTL_THREADS, 0, st>>>(d_sym, n, d_tab, p->sigma, wtiles, d_gcnt);
        HK_LAUNCH_CHECK();
        wt_tile_scan_kernel<<<p->sigma, 1024, 0, st>>>(d_gcnt, wtiles);
        HK_LAUNCH_CHECK();
        wt_levels_kernel<<<wtiles, WTL_THREADS, 0, st>>>(d_sym, n, d_tab, d_gcnt, wtiles, lw, p->levels, p->sigma);
        HK_LAUNCH_CHECK();
    }
    return wt_build_dirs(p, d_blob, dir, p->level_ones, st);
}

// Restoring a blob from stored level payloads (hkcsa_rrr_restore_level): _begin writes the node tables and clears the
// level regions, the caller ORs the payload bits in, _finish rebuilds block headers, superblocks, select samples and
// node counts and checks the ones per level against the plan.  Both sync.
extern "C" int hkcsa_wt_restore_begin(const hkcsa_wt_plan *p, void *d_blob, void *stream)
{
    HK_REQUIRE(p && d_blob, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_blob) & 31) == 0, HKCSA_EINVAL, "blob must be 32-byte aligned");
    cudaStream_t st = as_stream(stream);
    uint8_t *blob = static_cast<uint8_t *>(d_blob);
    int rc = wt_write_tables(p, blob, st);
    if (rc != HKCSA_OK) return rc;
    if (p->levels && p->blob_bytes > p->off_blocks[0])
        HK_CUDA(cudaMemsetAsync(blob + p->off_blocks[0], 0, p->blob_bytes - p->off_blocks[0], st));
    return HKCSA_OK;
}

extern "C" int hkcsa_wt_restore_finish(const hkcsa_wt_plan *p, void *d_blob, void *d_scratch, size_t scratch_bytes,
                                       void *stream)
{
    HK_REQUIRE(p && d_blob, HKCSA_EINVAL, "null pointer");
    if (p->levels == 0 || p->n == 0) return HKCSA_OK;
    HK_REQUIRE(d_scratch && p->scratch_bytes <= scratch_bytes, HKCSA_ESCRATCH, "wavelet scratch too small");
    Carver c(d_scratch);
    const DirScratch dir = carve_dir_scratch(c, p->n, HKCSA_MAX_LEVELS, WTC_BLOCKS_PER_CTA);
    uint64_t ones[HKCSA_MAX_LEVELS];
    int rc = wt_build_dirs(p, d_blob, dir, ones, as_stream(stream));
    if (rc != HKCSA_OK) return rc;
    for (uint32_t l = 0; l < p->levels; ++l)
        HK_REQUIRE(ones[l] == p->level_ones[l], HKCSA_EINVAL, "restored level holds a different number of ones than its plan");
    return HKCSA_OK;
}

#define HK_LEVEL_CHECK()                                                                              \
    HK_REQUIRE(h_plan && d_blob, HKCSA_EINVAL, "null pointer");                                        \
    HK_REQUIRE(level < h_plan->levels, HKCSA_EINVAL, "level out of range")

extern "C" int hkcsa_bv_rank_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                                   const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream)
{
    HK_LEVEL_CHECK();
    if (m == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    bv_rank_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(wt.level[level], d_pos, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_bv_select_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                                     const uint64_t *d_k, uint64_t m, uint64_t *d_out, void *stream)
{
    HK_LEVEL_CHECK();
    if (m == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    const uint32_t *samples =
        reinterpret_cast<const uint32_t *>(static_cast<const uint8_t *>(d_blob) + h_plan->off_select[level]);
    bv_select_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(
        wt.level[level], samples, h_plan->level_ones[level], d_k, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_bv_unpack(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level, uint64_t begin,
                               uint64_t count, uint8_t *d_out, void *stream)
{
    HK_LEVEL_CHECK();
    HK_REQUIRE(begin + count <= h_plan->level_len[level], HKCSA_EINVAL, "range beyond the level");
    if (count == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    bv_unpack_kernel<<<(uint32_t)((count + 255) / 256), 256, 0, as_stream(stream)>>>(wt.level[level], begin, count,
                                                                                     d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_bv_rank_range(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level, uint64_t begin,
                                   uint64_t count, uint32_t *d_out, void *stream)
{
    HK_LEVEL_CHECK();
    HK_REQUIRE(begin + count <= h_plan->level_len[level] + 1, HKCSA_EINVAL, "range beyond the level");
    if (count == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    bv_rank_range_kernel<<<(uint32_t)((count + 255) / 256), 256, 0, as_stream(stream)>>>(wt.level[level], begin,
                                                                                         count, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_wt_rank_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint8_t *d_sym,
                                   const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream)
{
    HK_REQUIRE(h_plan && d_blob, HKCSA_EINVAL, "null pointer");
    if (m == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    wt_rank_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(wt, d_sym, d_pos, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

extern "C" int hkcsa_wt_access_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint64_t *d_pos,
                                     uint64_t m, uint8_t *d_out, void *stream)
{
    HK_REQUIRE(h_plan && d_blob, HKCSA_EINVAL, "null pointer");
    if (m == 0) return HKCSA_OK;
    WtDev wt = make_wt_dev(d_blob, h_plan);
    wt_access_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(wt, d_pos, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// ------------------------------------------------------------------ stand-alone bit-vector
// SuccinctRankSelect(bitmap) (reference csa/wavelet_tree.py:5-25) outside a tree:
// a one-level plan whose level 0 is the bitmap, so hkcsa_bv_* apply unchanged.
namespace hkcsa {
__global__ void nonzero_lut_kernel(uint8_t *lut) { lut[threadIdx.x] = threadIdx.x ? 1 : 0; }
}  // namespace hkcsa

extern "C" int hkcsa_bitvec_plan(uint64_t nbits, hkcsa_wt_plan *p)
{
    HK_REQUIRE(p, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(nbits <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    memset(p, 0, sizeof(*p));
    memset(p->code_of_sym, 0xFF, sizeof(p->code_of_sym));
    memset(p->node_id, 0xFF, sizeof(p->node_id));
    p->n = nbits;
    p->sigma = 2;
    p->levels = 1;
    p->level_len[0] = nbits;
    p->level_nodes[0] = 1;
    wt_layout_blob(p);
    Carver c(nullptr);
    carve_dir_scratch(c, nbits, 1, WTP_BLOCKS_PER_CTA);
    c.take<uint8_t>(256);
    p->scratch_bytes = c.total();
    return HKCSA_OK;
}

extern "C" int hkcsa_bitvec_build(const uint8_t *d_bits, hkcsa_wt_plan *p, void *d_blob, void *d_scratch,
                                  size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(p && d_blob && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(p->levels == 1 && p->scratch_bytes <= scratch_bytes, HKCSA_ESCRATCH, "bit-vector scratch too small");
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_blob) & 31) == 0, HKCSA_EINVAL, "blob must be 32-byte aligned");
    HK_REQUIRE(d_bits || p->n == 0, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    const uint64_t n = p->n;
    uint8_t *blob = static_cast<uint8_t *>(d_blob);
    Carver c(d_scratch);
    const DirScratch dir = carve_dir_scratch(c, n, 1, WTP_BLOCKS_PER_CTA);
    uint8_t *d_lut = c.take<uint8_t>(256);
    nonzero_lut_kernel<<<1, 256, 0, st>>>(d_lut);
    HK_LAUNCH_CHECK();
    const DirLevels D = packed_dir(reinterpret_cast<RankBlock *>(blob + p->off_blocks[0]),
                                   reinterpret_cast<uint64_t *>(blob + p->off_super[0]),
                                   reinterpret_cast<uint32_t *>(blob + p->off_select[0]), n);
    const uint64_t nblocks = D.nblocks[0];
    {
        prof::Scope ps(st, prof::WT_PACK, n + n / 8);
        wt_pack_kernel<<<D.tile0[1], WTP_THREADS, 0, st>>>(d_bits, n, d_lut, D.blocks[0], nblocks, dir.agg);
        HK_LAUNCH_CHECK();
    }
    {
        prof::Scope ps(st, prof::WT_DIR, nblocks * 8);
        wt_dir_scan_all_kernel<<<1, 1024, 0, st>>>(D, dir.agg, dir.carry, dir.ones);
        HK_LAUNCH_CHECK();
        wt_dir_fix_all_kernel<WTP_BLOCKS_PER_CTA><<<(uint32_t)((nblocks + 255) / 256), 256, 0, st>>>(D, dir.carry);
        HK_LAUNCH_CHECK();
    }
    uint64_t *h_ones = reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(pinned_page()) + 3072);
    HK_CUDA(cudaMemcpyAsync(h_ones, dir.ones, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    p->level_ones[0] = h_ones[0];
    return HKCSA_OK;
}

// Stable bucket partition of a byte sequence by a host-supplied byte -> bucket
// table (255 = drop).  Used for the reference's next_text (the subsequence of
// symbols in the left half of the alphabet, csa/wavelet_tree.py:92).
// h_bucket_sizes[256] receives the element count of every bucket.  syncs.
extern "C" size_t hkcsa_partition_scratch_bytes(uint64_t n)
{
    Carver c(nullptr);
    c.take<uint64_t>(256);
    c.take<uint8_t>(256);
    c.take<uint32_t>(256);
    carve_sort_scratch(c, n);
    return c.total();
}

extern "C" int hkcsa_partition_bytes(const uint8_t *d_in, uint64_t n, const uint8_t *h_lut, uint8_t *d_out,
                                     uint64_t *h_bucket_sizes, void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(h_lut && h_bucket_sizes && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(n <= HKCSA_MAX_N, HKCSA_ERANGE, "n exceeds HKCSA_MAX_N");
    memset(h_bucket_sizes, 0, 256 * sizeof(uint64_t));
    if (n == 0) return HKCSA_OK;
    HK_REQUIRE(d_in && d_out, HKCSA_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    Carver c(d_scratch);
    uint64_t *d_hist = c.take<uint64_t>(256);
    uint8_t *d_lut = c.take<uint8_t>(256);
    uint32_t *d_base = c.take<uint32_t>(256);
    SortScratch ss = carve_sort_scratch(c, n);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "partition scratch too small");
    int rc = hkcsa_byte_hist(d_in, n, d_hist, stream);
    if (rc != HKCSA_OK) return rc;
    uint64_t *h_hist = reinterpret_cast<uint64_t *>(pinned_page());
    HK_CUDA(cudaMemcpyAsync(h_hist, d_hist, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < 256; ++b) h_bucket_sizes[h_lut[b]] += h_hist[b];
    uint32_t base[256];
    uint64_t run = 0;
    for (int k = 0; k < 256; ++k) { base[k] = (uint32_t)run; run += h_bucket_sizes[k]; }
    HK_CUDA(cudaMemcpyAsync(d_lut, h_lut, 256, cudaMemcpyHostToDevice, st));
    HK_CUDA(cudaMemcpyAsync(d_base, base, sizeof(base), cudaMemcpyHostToDevice, st));
    HK_CUDA(radix_partition_bytes(d_in, d_out, nullptr, (uint32_t)n, d_lut, d_base, ss, st));
    HK_CUDA(cudaStreamSynchronize(st));   // base[] lives on this stack frame
    return HKCSA_OK;
}
