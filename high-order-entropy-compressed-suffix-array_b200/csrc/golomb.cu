// golomb.cu -- Golomb-Rice run code of a level prefix.  Replaces
// GolombRiceEncoder.encode (reference csa/wavelet_tree.py:40-63): every maximal
// run of ones of length v, closed by a zero or by the end of input, emits
// v / m zeros, a one, then v % m as exactly m binary digits MSB first; runs of
// zeros emit nothing.  Output: one byte per code bit (the reference's list of
// 0/1 ints).  Low priority on the path (feeds only WaveletTree.compress), so
// the kernels are simple: one thread walks one 1792-bit chunk; runs that cross
// chunk boundaries are stitched by a scan of (trailing ones, all-ones) pairs.
#include "common.cuh"
#include "wavelet.cuh"

namespace hkcsa {

constexpr uint32_t G_BLOCKS = 8;
constexpr uint32_t G_BITS = G_BLOCKS * HKCSA_BLOCK_BITS;   // 1792
constexpr uint32_t G_ALL = 1u << 31;

struct ChunkWalker {
    const BitVec &v;
    uint64_t lo, hi;
    __device__ ChunkWalker(const BitVec &bv, uint64_t chunk, uint64_t nbits)
        : v(bv), lo(chunk * G_BITS), hi(min(nbits, (chunk + 1) * (uint64_t)G_BITS)) {}
    template <typename F>
    __device__ void for_each_bit(F f) const
    {
        for (uint64_t g = lo / HKCSA_BLOCK_BITS; g * HKCSA_BLOCK_BITS < hi; ++g) {
            const RankBlock b = load_block(v.blocks + g);
            const uint64_t w[4] = {b.w[0], b.w[1], b.w[2], b.w[3]};
            const uint32_t cnt = (uint32_t)min((uint64_t)HKCSA_BLOCK_BITS, hi - g * HKCSA_BLOCK_BITS);
            for (uint32_t o = 0; o < cnt; ++o) {
                const uint32_t t = o + 32u;
                const uint64_t word = (t < 64) ? w[0] : (t < 128) ? w[1] : (t < 192) ? w[2] : w[3];
                f((uint32_t)(word >> (t & 63u)) & 1u);
            }
        }
    }
};

// tail[c] = trailing ones of chunk c, | G_ALL when the whole chunk is ones
__global__ void golomb_tail_kernel(BitVec v, uint64_t nbits, uint64_t chunks, uint32_t *__restrict__ tail)
{
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= chunks) return;
    ChunkWalker w(v, c, nbits);
    uint32_t run = 0, len = 0;
    bool all = true;
    w.for_each_bit([&](uint32_t bit) {
        ++len;
        if (bit) ++run; else { run = 0; all = false; }
    });
    tail[c] = run | (all ? G_ALL : 0u);
    (void)len;
}

// carry[c] = ones immediately preceding chunk c: exclusive scan of (tail, all) under
// (t1,a1)+(t2,a2) = (a2 ? t1+t2 : t2, a1&&a2), identity (0, all).  On the tail[] words: the flag of a sum is the
// left one's when the right one is all ones (a run is at most 2^30 bits, the count never reaches the flag).
// Single CTA.
__global__ void __launch_bounds__(1024)
golomb_carry_kernel(const uint32_t *__restrict__ tail, uint64_t chunks, uint32_t *__restrict__ carry)
{
    block_excl_scan_carried(chunks, G_ALL, [](uint32_t a, uint32_t b) { return (b & G_ALL) ? a + (b & ~G_ALL) : b; },
                            [&](uint64_t c) { return tail[c]; }, [&](uint64_t c, uint32_t p) { carry[c] = p & ~G_ALL; });
}

// off[c] = code bits of the chunks before c, *total = all of them.  Single CTA.
__global__ void __launch_bounds__(1024)
golomb_off_kernel(const uint32_t *__restrict__ len, uint64_t chunks, uint64_t *__restrict__ off, uint64_t *__restrict__ total)
{
    const uint64_t t = block_excl_scan_carried(chunks, (uint64_t)0, Plus(), [&](uint64_t c) { return (uint64_t)len[c]; },
                                               [&](uint64_t c, uint64_t p) { off[c] = p; });
    if (threadIdx.x == 0) *total = t;
}

template <bool EMIT>
__global__ void golomb_emit_kernel(BitVec v, uint64_t nbits, uint64_t chunks, uint32_t m,
                                   const uint32_t *__restrict__ carry, uint32_t *__restrict__ len_out,
                                   const uint64_t *__restrict__ off, uint8_t *__restrict__ out)
{
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= chunks) return;
    ChunkWalker w(v, c, nbits);
    uint64_t q = carry[c];
    uint64_t written = 0;
    uint8_t *dst = EMIT ? out + off[c] : nullptr;
    auto flush = [&]() {
        const uint64_t quo = q / m, rem = q % m;
        if (EMIT) {
            for (uint64_t z = 0; z < quo; ++z) dst[written + z] = 0;
            dst[written + quo] = 1;
            for (uint32_t b = 0; b < m; ++b) {
                const uint32_t sh = m - 1 - b;
                dst[written + quo + 1 + b] = (sh < 64) ? (uint8_t)((rem >> sh) & 1u) : (uint8_t)0;
            }
        }
        written += quo + 1 + m;
        q = 0;
    };
    w.for_each_bit([&](uint32_t bit) {
        if (bit) ++q;
        else if (q > 0) flush();
    });
    if (c == chunks - 1 && q > 0) flush();   // end of input closes the last run
    if (!EMIT) len_out[c] = (uint32_t)written;
}

}  // namespace hkcsa

using namespace hkcsa;

namespace {
struct GolombScratch {
    uint32_t *tail, *carry, *len;
    uint64_t *off, *total;
};
GolombScratch carve_golomb(Carver &c, uint64_t nbits)
{
    const uint64_t chunks = (nbits + G_BITS - 1) / G_BITS + 1;
    GolombScratch g;
    g.tail = c.take<uint32_t>(chunks);
    g.carry = c.take<uint32_t>(chunks);
    g.len = c.take<uint32_t>(chunks);
    g.off = c.take<uint64_t>(chunks);
    g.total = c.take<uint64_t>(8);
    return g;
}
}  // namespace

extern "C" size_t hkcsa_golomb_scratch_bytes(uint64_t nbits)
{
    Carver c(nullptr);
    carve_golomb(c, nbits);
    return c.total();
}

extern "C" int hkcsa_golomb_encode(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level, uint64_t nbits,
                                   uint32_t m, uint8_t *d_out, uint64_t out_capacity, uint64_t *h_out_bits,
                                   void *d_scratch, size_t scratch_bytes, void *stream)
{
    HK_REQUIRE(h_plan && d_blob && h_out_bits && d_scratch, HKCSA_EINVAL, "null pointer");
    HK_REQUIRE(level < h_plan->levels, HKCSA_EINVAL, "level out of range");
    HK_REQUIRE(nbits <= h_plan->level_len[level], HKCSA_EINVAL, "nbits beyond the level");
    HK_REQUIRE(m >= 1 && m <= 62, HKCSA_EINVAL, "m out of range");
    *h_out_bits = 0;
    if (nbits == 0) return HKCSA_OK;
    Carver c(d_scratch);
    GolombScratch g = carve_golomb(c, nbits);
    HK_REQUIRE(c.total() <= scratch_bytes, HKCSA_ESCRATCH, "golomb scratch too small");
    cudaStream_t st = as_stream(stream);
    WtDev wt = make_wt_dev(d_blob, h_plan);
    const BitVec v = wt.level[level];
    const uint64_t chunks = (nbits + G_BITS - 1) / G_BITS;
    const uint32_t grid = (uint32_t)((chunks + 127) / 128);
    golomb_tail_kernel<<<grid, 128, 0, st>>>(v, nbits, chunks, g.tail);
    HK_LAUNCH_CHECK();
    golomb_carry_kernel<<<1, 1024, 0, st>>>(g.tail, chunks, g.carry);
    HK_LAUNCH_CHECK();
    golomb_emit_kernel<false><<<grid, 128, 0, st>>>(v, nbits, chunks, m, g.carry, g.len, nullptr, nullptr);
    HK_LAUNCH_CHECK();
    golomb_off_kernel<<<1, 1024, 0, st>>>(g.len, chunks, g.off, g.total);
    HK_LAUNCH_CHECK();
    uint64_t *h_total = reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(pinned_page()) + 3584);
    HK_CUDA(cudaMemcpyAsync(h_total, g.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HK_CUDA(cudaStreamSynchronize(st));
    *h_out_bits = *h_total;
    if (d_out == nullptr) return HKCSA_OK;
    HK_REQUIRE(out_capacity >= *h_total, HKCSA_ESCRATCH, "golomb output buffer too small");
    golomb_emit_kernel<true><<<grid, 128, 0, st>>>(v, nbits, chunks, m, g.carry, nullptr, g.off, d_out);
    HK_LAUNCH_CHECK();
    return HKCSA_OK;
}
