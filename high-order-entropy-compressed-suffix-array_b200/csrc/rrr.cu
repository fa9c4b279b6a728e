// rrr.cu -- entropy-coded bit-vectors with rank on the coded form (SURVEY.md section 8f, row 3).
//
// The reference's compress() keeps Golomb run codes that cannot be decoded (zero runs are not coded:
// csa/wavelet_tree.py:40-63; its decompress() returns '', :158-200).  This is the lossless counterpart: the
// class/offset code of Raman-Raman-Rao with 15-bit blocks, which stores a bit-vector in n*H_0 + o(n) bits -- applied to
// the wavelet-tree levels of a BWT that is what makes the index "high-order entropy compressed" (n*H_k + o(n)).
//
//   block b (15 bits)   class c = popcount (4 bits, packed two per byte)
//                       offset  = index of the 15-bit pattern among the C(15, c) patterns of its class,
//                                 ceil(log2 C(15, c)) bits in one bit stream
//   superblock (64 blocks = 960 bits)  {ones before it, bit position of its first offset}: 2 x 32 bits
//
// rank(i) reads one superblock entry, the 32 class bytes of the superblock (one sector), one offset and one table
// entry -- it never expands the vector.  decode restores the level payload bit for bit (save / load round trip).
#include "common.cuh"
#include "prof.cuh"
#include "wavelet.cuh"
#include <mutex>

namespace hkcsa {

constexpr uint32_t RRR_B = 15;
constexpr uint32_t RRR_SB = 64;                       // blocks per superblock
constexpr uint32_t RRR_SB_BITS = RRR_B * RRR_SB;      // 960

// ceil(log2 C(15, c)) for c = 0..15, four bits each: 0 4 7 9 11 12 13 13 13 13 12 11 9 7 4 0
constexpr uint64_t RRR_CLS_BITS = 0x0479BCDDDDCB9740ull;
__host__ __device__ __forceinline__ uint32_t rrr_cls_bits(uint32_t c) { return (uint32_t)(RRR_CLS_BITS >> (4 * c)) & 15u; }

struct RrrTables {
    uint16_t pattern[32768];      // patterns ordered by (class, value)
    uint16_t offset_of[32768];    // pattern -> index inside its class
    uint16_t cls_start[17];
    uint8_t cls_bits[16];
};

struct RrrSuper {                 // 8 bytes per 960 bits (a vector holds at most HKCSA_MAX_N < 2^30 bits)
    uint32_t ones;                // ones before the superblock
    uint32_t bitpos;              // position of the superblock's first offset in the stream
};

struct RrrDev {
    const RrrSuper *super;
    const uint8_t *classes;       // two per byte, low nibble first
    const uint32_t *stream;
    uint64_t nbits, nblocks;
};

// `cnt` (<= 32) payload bits of a level starting at bit j (bits past `len` read as 0)
__device__ __forceinline__ uint32_t level_bits(const RankBlock *__restrict__ blocks, uint64_t len, uint64_t j, uint32_t cnt)
{
    if (j >= len) return 0u;
    const uint64_t rb = j / HKCSA_BLOCK_BITS;
    const uint32_t o = (uint32_t)(j - rb * HKCSA_BLOCK_BITS);
    const uint32_t t = 32u + o, w = t >> 6, r = t & 63u;
    const uint64_t *q = blocks[rb].w;
    uint64_t v = q[w] >> r;
    if (r + cnt > 64u && w < 3u) v |= q[w + 1] << (64u - r);
    const uint32_t avail = HKCSA_BLOCK_BITS - o;
    if (cnt > avail && (rb + 1) * (uint64_t)HKCSA_BLOCK_BITS < len) v |= (blocks[rb + 1].w[0] >> 32) << avail;
    uint32_t out = (uint32_t)v & (cnt >= 32u ? 0xFFFFFFFFu : ((1u << cnt) - 1u));
    if (j + cnt > len) out &= (1u << (uint32_t)(len - j)) - 1u;
    return out;
}

__device__ __forceinline__ uint32_t stream_get(const uint32_t *__restrict__ s, uint64_t bitpos, uint32_t cnt)
{
    if (cnt == 0) return 0u;
    const uint64_t w = bitpos >> 5;
    const uint32_t r = (uint32_t)(bitpos & 31u);
    uint64_t v = s[w];
    if (r + cnt > 32u) v |= (uint64_t)s[w + 1] << 32;
    return (uint32_t)(v >> r) & ((1u << cnt) - 1u);
}
__device__ __forceinline__ void stream_put(uint32_t *s, uint64_t bitpos, uint32_t cnt, uint32_t val)
{
    if (cnt == 0) return;
    const uint64_t w = bitpos >> 5;
    const uint32_t r = (uint32_t)(bitpos & 31u);
    atomicOr(&s[w], val << r);
    if (r + cnt > 32u) atomicOr(&s[w + 1], val >> (32u - r));
}

// pass 1: ones and offset bits of every superblock
__global__ void __launch_bounds__(256)
rrr_size_kernel(const RankBlock *__restrict__ blocks, uint64_t nbits, uint64_t nsuper, const RrrTables *__restrict__ T,
                uint64_t *__restrict__ sb_ones, uint64_t *__restrict__ sb_bits)
{
    const uint64_t sb = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (sb >= nsuper) return;
    uint32_t ones = 0, bits = 0;
    for (uint32_t b = 0; b < RRR_SB; ++b) {
        const uint32_t c = __popc(level_bits(blocks, nbits, (sb * RRR_SB + b) * RRR_B, RRR_B));
        ones += c;
        bits += rrr_cls_bits(c);
    }
    sb_ones[sb] = ones;
    sb_bits[sb] = bits;
}

// single CTA: exclusive scans of both rows into the superblock table; totals -> tot[0] (ones), tot[1] (stream bits)
struct RrrSums {
    uint64_t ones, bits;
};
__global__ void __launch_bounds__(1024)
rrr_scan_kernel(const uint64_t *__restrict__ sb_ones, const uint64_t *__restrict__ sb_bits, uint64_t nsuper,
                RrrSuper *__restrict__ super, uint64_t *__restrict__ tot)
{
    const RrrSums t = block_excl_scan_carried(
        nsuper, RrrSums{0, 0}, [](RrrSums a, RrrSums b) { return RrrSums{a.ones + b.ones, a.bits + b.bits}; },
        [&](uint64_t i) { return RrrSums{sb_ones[i], sb_bits[i]}; },
        [&](uint64_t i, RrrSums p) { super[i] = RrrSuper{(uint32_t)p.ones, (uint32_t)p.bits}; });
    if (threadIdx.x == 0) { tot[0] = t.ones; tot[1] = t.bits; }
}

// pass 2: classes (a thread owns the 32 class bytes of its superblock) and offsets (shared words: atomicOr)
__global__ void __launch_bounds__(256)
rrr_emit_kernel(const RankBlock *__restrict__ blocks, uint64_t nbits, uint64_t nsuper, const RrrTables *__restrict__ T,
                const RrrSuper *__restrict__ super, uint8_t *__restrict__ classes, uint32_t *__restrict__ stream)
{
    const uint64_t sb = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (sb >= nsuper) return;
    uint64_t bitpos = super[sb].bitpos;
    for (uint32_t b = 0; b < RRR_SB; b += 2) {
        uint32_t byte = 0;
        for (uint32_t h = 0; h < 2; ++h) {
            const uint32_t pat = level_bits(blocks, nbits, (sb * RRR_SB + b + h) * RRR_B, RRR_B);
            const uint32_t c = __popc(pat), nb = rrr_cls_bits(c);
            byte |= c << (4 * h);
            stream_put(stream, bitpos, nb, T->offset_of[pat]);
            bitpos += nb;
        }
        classes[sb * (RRR_SB / 2) + b / 2] = (uint8_t)byte;
    }
}

// class of block `blk`, the position of its offset, and the ones before it
__device__ __forceinline__ uint32_t rrr_seek(const RrrDev &v, uint64_t blk, uint64_t &ones, uint64_t &bitpos)
{
    const uint64_t sb = blk / RRR_SB;
    const uint32_t in = (uint32_t)(blk - sb * RRR_SB);
    const RrrSuper su = v.super[sb];
    const uint4 *cp = reinterpret_cast<const uint4 *>(v.classes + sb * (RRR_SB / 2));      // 32 bytes: one sector
    const uint4 q0 = __ldg(cp), q1 = __ldg(cp + 1);
    const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    uint32_t cls = 0, o = 0, bp = 0;
#pragma unroll
    for (uint32_t b = 0; b < RRR_SB; ++b) {
        const uint32_t c = (w[b >> 3] >> (4 * (b & 7u))) & 15u;
        if (b < in) { o += c; bp += rrr_cls_bits(c); }
        if (b == in) cls = c;
    }
    ones = su.ones + o;
    bitpos = su.bitpos + bp;
    return cls;
}
__device__ __forceinline__ uint32_t rrr_block(const RrrDev &v, const RrrTables *__restrict__ T, uint32_t c, uint64_t bitpos)
{
    return T->pattern[T->cls_start[c] + stream_get(v.stream, bitpos, rrr_cls_bits(c))];
}

__global__ void rrr_rank_kernel(RrrDev v, const RrrTables *__restrict__ T, const uint64_t *__restrict__ pos, uint64_t m,
                                uint64_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const uint64_t i = min(pos[q], v.nbits);
    const uint64_t blk = i / RRR_B;
    const uint32_t o = (uint32_t)(i - blk * RRR_B);
    if (blk >= v.nblocks) {            // i == nbits on a block boundary: everything before the end
        uint64_t ones, bitpos;
        const uint32_t c = rrr_seek(v, v.nblocks - 1, ones, bitpos);
        out[q] = ones + c;
        return;
    }
    uint64_t ones, bitpos;
    const uint32_t c = rrr_seek(v, blk, ones, bitpos);
    out[q] = ones + (o ? __popc(rrr_block(v, T, c, bitpos) & ((1u << o) - 1u)) : 0u);
}

// bits [begin, begin + count) as one byte per bit
__global__ void rrr_unpack_kernel(RrrDev v, const RrrTables *__restrict__ T, uint64_t begin, uint64_t count,
                                  uint8_t *__restrict__ out)
{
    const uint64_t first = begin / RRR_B;
    const uint64_t blk = first + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= v.nblocks || blk * RRR_B >= begin + count) return;
    uint64_t ones, bitpos;
    const uint32_t c = rrr_seek(v, blk, ones, bitpos);
    const uint32_t pat = rrr_block(v, T, c, bitpos);
    for (uint32_t t = 0; t < RRR_B; ++t) {
        const uint64_t j = blk * RRR_B + t;
        if (j >= begin && j < begin + count && j < v.nbits) out[j - begin] = (uint8_t)((pat >> t) & 1u);
    }
}

// the whole vector back into the payload bits of a level's rank blocks (which must be zero)
__global__ void rrr_restore_kernel(RrrDev v, const RrrTables *__restrict__ T, uint32_t *__restrict__ level_words)
{
    const uint64_t blk = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= v.nblocks) return;
    uint64_t ones, bitpos;
    const uint32_t c = rrr_seek(v, blk, ones, bitpos);
    uint32_t pat = rrr_block(v, T, c, bitpos);
    while (pat) {
        const uint32_t t = __ffs(pat) - 1;
        pat &= pat - 1;
        const uint64_t j = blk * RRR_B + t;
        const uint64_t rb = j / HKCSA_BLOCK_BITS;
        const uint32_t bit = 32u + (uint32_t)(j - rb * HKCSA_BLOCK_BITS);
        atomicOr(&level_words[rb * 8 + (bit >> 5)], 1u << (bit & 31u));
    }
}

static RrrDev make_rrr_dev(const void *d_rrr, const hkcsa_rrr_plan *p)
{
    const uint8_t *b = static_cast<const uint8_t *>(d_rrr);
    RrrDev v;
    v.super = reinterpret_cast<const RrrSuper *>(b + p->off_super);
    v.classes = b + p->off_classes;
    v.stream = reinterpret_cast<const uint32_t *>(b + p->off_stream);
    v.nbits = p->nbits;
    v.nblocks = p->nblocks;
    return v;
}

static void rrr_layout(hkcsa_rrr_plan *p, uint64_t nbits, uint64_t ones, uint64_t stream_bits)
{
    memset(p, 0, sizeof(*p));
    p->nbits = nbits;
    p->nblocks = (nbits + RRR_B - 1) / RRR_B;
    p->nsuper = (p->nblocks + RRR_SB - 1) / RRR_SB;
    p->ones = ones;
    p->stream_bits = stream_bits;
    uint64_t off = 0;
    p->off_super = off;
    off = align_up(off + (p->nsuper + 1) * sizeof(RrrSuper), 256);
    p->off_classes = off;
    off = align_up(off + (p->nsuper + 1) * (RRR_SB / 2), 256);
    p->off_stream = off;
    off = align_up(off + ((stream_bits + 31) / 32 + 2) * sizeof(uint32_t), 256);
    p->blob_bytes = off;
}

}  // namespace hkcsa

using namespace hkcsa;

extern "C" size_t hkcsa_rrr_tables_bytes(void) { return sizeof(RrrTables); }

// writes the class / offset tables (a pure function of the block size) to d_tables.  syncs.
extern "C" int hkcsa_rrr_tables_init(void *d_tables, void *stream)
{
    HK_REQUIRE(d_tables != nullptr, HKCSA_EINVAL, "null pointer");
    static RrrTables T;
    static bool ready = false;
    static std::mutex mu;
    {
        std::lock_guard<std::mutex> lock(mu);
        if (!ready) {
            uint32_t at = 0;
            for (uint32_t c = 0; c <= RRR_B; ++c) {
                T.cls_start[c] = (uint16_t)at;
                uint32_t k = 0;
                for (uint32_t pat = 0; pat < 32768u; ++pat)
                    if ((uint32_t)__builtin_popcount(pat) == c) {
                        T.pattern[at + k] = (uint16_t)pat;
                        T.offset_of[pat] = (uint16_t)k;
                        ++k;
                    }
                at += k;
                uint8_t bits = 0;
                while ((1u << bits) < k) ++bits;
                T.cls_bits[c] = bits;
                if (bits != rrr_cls_bits(c)) { set_error("rrr class widths disagree"); return HKCSA_EINVAL; }
            }
            T.cls_start[16] = (uint16_t)at;      // 32768 wraps to 0: never read
            ready = true;
        }
    }
    cudaStream_t st = as_stream(stream);
    HK_CUDA(cudaMemcpyAsync(d_tables, &T, sizeof(T), cudaMemcpyHostToDevice, st));
    HK_CUDA(cudaStreamSynchronize(st));
    return HKCSA_OK;
}

extern "C" size_t hkcsa_rrr_scratch_bytes(uint64_t nbits)
{
    Carver c(nullptr);
    const uint64_t nsuper = (nbits + RRR_SB_BITS - 1) / RRR_SB_BITS + 1;
    c.take<uint64_t>(nsuper);
    c.take<uint64_t>(nsuper);
    c.take<uint64_t>(4);
    c.take<RrrSuper>(nsuper);
    return c.total();
}

// Encodes bits [0, nbits) of `level` of a wavelet-tree blob.  Two calls: d_out == NULL sizes the code (fills
// *h_plan), otherwise writes it (h_plan->blob_bytes bytes, 32-byte aligned).  syncs.
extern "C" int hkcsa_rrr_encode(const void *d_wt_blob, const hkcsa_wt_plan *h_wt, uint32_t level, uint64_t nbits,
                                const void *d_tables, hkcsa_rrr_plan *h_plan, void *d_out, size_t out_capacity,
                                void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(d_wt_blob && h_wt && d_tables && h_plan && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(level < h_wt->levels && nbits <= h_wt->level_len[level], HKCSA_EINVAL, "level / nbits out of range");
    HK_REQUIRE(nbits <= HKCSA_MAX_N + 1, HKCSA_ERANGE, "vector exceeds HKCSA_MAX_N bits (32-bit superblock entries)");
    HK_REQUIRE(!d_out || (reinterpret_cast<uintptr_t>(d_out) & 31) == 0, HKCSA_EINVAL, "output must be 32-byte aligned");
    cudaStream_t st = as_stream(stream);
    rrr_layout(h_plan, nbits, 0, 0);
    if (nbits == 0) return HKCSA_OK;
    const uint64_t nsuper = h_plan->nsuper;
    Carver c(d_scratch);
    uint64_t *sb_ones = c.take<uint64_t>(nsuper + 1);
    uint64_t *sb_bits = c.take<uint64_t>(nsuper + 1);
    uint64_t *d_tot = c.take<uint64_t>(4);
    RrrSuper *tmp_super = c.take<RrrSuper>(nsuper + 1);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "rrr scratch too small");
    const RankBlock *blocks = reinterpret_cast<const RankBlock *>(static_cast<const uint8_t *>(d_wt_blob) + h_wt->off_blocks[level]);
    const RrrTables *T = static_cast<const RrrTables *>(d_tables);
    const uint32_t grid = (uint32_t)((nsuper + 255) / 256);
    prof::Scope ps(st, prof::OTHER, nbits / 4);
    rrr_size_kernel<<<grid, 256, 0, st>>>(blocks, nbits, nsuper, T, sb_ones, sb_bits);
    HK_LAUNCH_CHECK();
    if (d_out) HK_CUDA(cudaMemsetAsync(d_out, 0, out_capacity, st));      // offsets are OR-ed into the stream
    RrrSuper *super_dst = d_out ? reinterpret_cast<RrrSuper *>(d_out) : tmp_super;   // off_super == 0
    HK_REQUIRE(!d_out || out_capacity >= (nsuper + 1) * sizeof(RrrSuper), HKCSA_ESCRATCH, "rrr output too small");
    rrr_scan_kernel<<<1, 1024, 0, st>>>(sb_ones, sb_bits, nsuper, super_dst, d_tot);
    HK_LAUNCH_CHECK();
    uint64_t h_tot[2];
    HK_CUDA(cudaMemcpyAsync(h_tot, d_tot, sizeof(h_tot), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    rrr_layout(h_plan, nbits, h_tot[0], h_tot[1]);
    if (!d_out) return HKCSA_OK;
    HK_REQUIRE(h_plan->blob_bytes <= out_capacity, HKCSA_ESCRATCH, "rrr output too small");
    uint8_t *ob = static_cast<uint8_t *>(d_out);
    rrr_emit_kernel<<<grid, 256, 0, st>>>(blocks, nbits, nsuper, T, super_dst, ob + h_plan->off_classes,
                                          reinterpret_cast<uint32_t *>(ob + h_plan->off_stream));
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

#define HK_RRR_CHECK()                                                                              \
    HK_REQUIRE(d_rrr && h_plan && d_tables, HKCSA_EINVAL, "null pointer");                           \
    HK_REQUIRE((reinterpret_cast<uintptr_t>(d_rrr) & 31) == 0, HKCSA_EINVAL, "coded vector must be 32-byte aligned")

// rank(i) = ones in bits [0, i) on the coded form, i clamped to nbits
extern "C" int hkcsa_rrr_rank_batch(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables,
                                    const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream)
{
    if (m == 0) return HKCSA_OK;
    HK_RRR_CHECK();
    HK_REQUIRE(d_pos && d_out, HKCSA_EINVAL, "null pointer");
    if (h_plan->nbits == 0) { HK_CUDA(cudaMemsetAsync(d_out, 0, m * sizeof(uint64_t), as_stream(stream))); return HKCSA_OK; }
    rrr_rank_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, as_stream(stream)>>>(make_rrr_dev(d_rrr, h_plan),
        static_cast<const RrrTables *>(d_tables), d_pos, m, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// bits [begin, begin + count) decoded to one byte per bit
extern "C" int hkcsa_rrr_unpack(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables, uint64_t begin,
                                uint64_t count, uint8_t *d_out, void *stream)
{
    if (count == 0) return HKCSA_OK;
    HK_RRR_CHECK();
    HK_REQUIRE(d_out && begin + count <= h_plan->nbits, HKCSA_EINVAL, "range");
    const uint64_t nblk = (begin + count + RRR_B - 1) / RRR_B - begin / RRR_B;
    rrr_unpack_kernel<<<(uint32_t)((nblk + 255) / 256), 256, 0, as_stream(stream)>>>(make_rrr_dev(d_rrr, h_plan),
        static_cast<const RrrTables *>(d_tables), begin, count, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}

// Decodes the vector into the payload bits of `level` of a wavelet-tree blob (the level region must be zero:
// hkcsa_wt_restore_begin clears it); hkcsa_wt_restore_finish then rebuilds the block headers and directories.
extern "C" int hkcsa_rrr_restore_level(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables,
                                       const hkcsa_wt_plan *h_wt, uint32_t level, void *d_wt_blob, void *stream)
{
    HK_RRR_CHECK();
    HK_REQUIRE(h_wt && d_wt_blob && level < h_wt->levels, HKCSA_EINVAL, "bad level");
    HK_REQUIRE(h_plan->nbits == h_wt->level_len[level], HKCSA_EINVAL, "coded vector and level lengths differ");
    if (h_plan->nbits == 0) return HKCSA_OK;
    uint32_t *words = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(d_wt_blob) + h_wt->off_blocks[level]);
    prof::Scope ps(as_stream(stream), prof::OTHER, h_plan->nbits / 4);
    rrr_restore_kernel<<<(uint32_t)((h_plan->nblocks + 255) / 256), 256, 0, as_stream(stream)>>>(
        make_rrr_dev(d_rrr, h_plan), static_cast<const RrrTables *>(d_tables), words);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
