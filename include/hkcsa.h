/*
 * hkcsa.h -- C-ABI of libhkcsa.so: the B200 (sm_100a) hot path of the H_k-CSA
 * index: suffix array -> BWT -> wavelet tree with rank/select directories, and
 * batched FM backward search (count / locate).
 *
 * The reference (ajaynair710/High-Order-Entropy-Compressed-Suffix-Array) is pure
 * Python and has no FFI layer of its own (SURVEY.md section 8b): these entry
 * points are what the reference's Python functions bind to through ctypes when
 * its csa/*.py modules are swapped for ours (INTEGRATION.md shows the stub).
 * Each entry point cites the reference function it replaces (file:line relative
 * to the reference repository root).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes.  No exceptions cross the boundary.
 *  - Every function returns an int status: HKCSA_OK (0) or a negative HKCSA_E*;
 *    hkcsa_last_error() returns a thread-local message for the last failure.
 *  - Pointers prefixed d_ are DEVICE pointers, h_ are HOST pointers.  The
 *    caller allocates every device buffer, scratch included (sizes come from
 *    the *_bytes queries); the library allocates no device memory.  Its only
 *    allocation is one small pinned host page per calling thread for scalar read-backs.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *    Work is enqueued on that stream.  Functions documented as "syncs" wait on
 *    the stream because they return scalars to the host; all others are async.
 *  - Symbols are bytes (latin-1 text: utils/data_loader.py:4), ordered as
 *    unsigned bytes == Python code-point order.  Text length n <= HKCSA_MAX_N.
 */
#ifndef HKCSA_H
#define HKCSA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HKCSA_OK        0
#define HKCSA_EINVAL   (-1)  /* bad argument                                   */
#define HKCSA_ECUDA    (-2)  /* CUDA runtime error (see hkcsa_last_error)      */
#define HKCSA_ESCRATCH (-3)  /* scratch / output buffer too small              */
#define HKCSA_ERANGE   (-4)  /* n exceeds HKCSA_MAX_N                          */

#define HKCSA_MAX_N ((uint64_t)((1u << 30) - 2))
#define HKCSA_MAX_LEVELS 8
#define HKCSA_ABI_VERSION 1

int         hkcsa_abi_version(void);
const char *hkcsa_last_error(void);
/* sizeof of the public structs (0 hkcsa_sa_stats, 1 hkcsa_wt_plan, 2 hkcsa_ssa_plan, */
/* 3 hkcsa_prof_entry, 4 hkcsa_occ_plan, 5 hkcsa_dsa_plan, 6 hkcsa_rrr_plan) so a    */
/* binding can verify its mirror.                                                     */
size_t      hkcsa_struct_size(int which);

/* ------------------------------------------------------------------------ */
/* Workload synthesis (bench/tests; no reference counterpart -- the corpus    */
/* URLs of tests/dataset_benchmark.py:10-16 are unreachable offline).         */
/* kind: 0 = ENG96 order-3 Markov English-like, 1 = DNA4 order-5 Markov.      */
/* ------------------------------------------------------------------------ */
int hkcsa_gen_text(int kind, uint64_t seed, uint64_t n, uint8_t *d_text, void *stream);
/* Patterns (semantics of tests/test_patterns.py:3-9, seeded): lengths first,  */
/* the caller prefix-sums them into d_offsets[P+1], then the bytes.            */
int hkcsa_gen_pattern_lengths(uint64_t seed, uint64_t P, uint32_t min_len, uint32_t max_len,
                              uint64_t n, uint32_t *d_len, void *stream);
int hkcsa_gen_pattern_bytes(uint64_t seed, uint64_t P, const uint8_t *d_text, uint64_t n,
                            const uint8_t *d_alphabet, uint32_t sigma, const int64_t *d_offsets,
                            uint8_t *d_out, void *stream);

/* ------------------------------------------------------------------------ */
/* K1  suffix array -- replaces build_suffix_array, csa/suffix_array.py:131-134*/
/*     (and the intent of ksa, :46-129).  Prefix doubling over packed 64-bit   */
/*     keys sorted by an LSD onesweep radix sort; suffixes whose rank is       */
/*     already unique leave the working set.  Proper prefixes sort first.      */
/* ------------------------------------------------------------------------ */
typedef struct hkcsa_sa_stats {
    uint32_t rounds;            /* doubling rounds executed (round 0 included)  */
    uint32_t bits_per_symbol;   /* b: width of a dense symbol code in round 0   */
    uint32_t k0;                /* symbols packed per key in round 0            */
    uint32_t sigma;             /* distinct bytes in the text                   */
    uint64_t sort_elem_passes;  /* sum over rounds of elements * radix passes   */
    uint64_t alg_bytes;         /* algorithmic HBM bytes moved (DESIGN.md K1)   */
    uint64_t round_elems[40];   /* working-set size per round                   */
    uint32_t round_passes[40];  /* radix passes per round                       */
    uint64_t byte_hist[256];    /* occurrences per byte value (the BWT has the  */
                                /* same histogram: hkcsa_wt_plan_from_hist)     */
    uint32_t key_bits0;         /* sorted bits of a round-0 key                 */
    uint32_t bwt_carried;       /* 1: the BWT came out of the round-0 sort      */
    uint32_t gram_k;            /* round-0 keys coded over k-grams (0: symbols) */
    uint32_t lazy_ranks;        /* 1: round 0 scattered no ranks; later rounds  */
                                /* look them up in the sorted round-0 keys      */
} hkcsa_sa_stats;

size_t hkcsa_sa_scratch_bytes(uint64_t n);
/* syncs (once per doubling round).  d_sa: uint32[n].  h_stats may be NULL.    */
int hkcsa_sa_build(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, void *d_scratch,
                   size_t scratch_bytes, void *stream, hkcsa_sa_stats *h_stats);

/* LSD onesweep radix sort of (uint64 key, uint32 value) pairs on the low       */
/* `key_bits` bits -- the primitive under K1, exported for tests/bench.         */
/* Result lands in (d_keys, d_vals); *_alt are same-sized ping-pong buffers.    */
size_t hkcsa_sort_scratch_bytes(uint64_t n);
int hkcsa_sort_pairs_u64(uint64_t *d_keys, uint32_t *d_vals, uint64_t *d_keys_alt, uint32_t *d_vals_alt,
                         uint64_t n, int key_bits, void *d_scratch, size_t scratch_bytes, void *stream);

/* Distributed build (BASELINE config 5: a text beyond one GPU's working set; no reference counterpart -- the   */
/* reference is single-process, but its build_suffix_array, csa/suffix_array.py:131-134, sorts ANY text and so   */
/* does this).  One process per GPU, up to HKCSA_DSA_MAX_RANKS ranks.  The text is replicated (one all-gather);  */
/* rank r keys the suffixes of ITS block of positions, and the kernel that packs the keys stores every (key, id) */
/* straight into the receive arrays of the rank owning the key's bucket through peer-mapped pointers (the        */
/* all-to-all bucket exchange is part of the pack kernel).  Each rank sorts what it received and refines its      */
/* groups: extension rounds read the next symbols from the replicated text; whatever survives them (repetitive    */
/* texts) is finished by rank doubling over the ranks' peer-mapped ISA blocks.  The slices concatenated in rank   */
/* order are the suffix array.  Suffix ids are uint32 up to n = 2^32-2 and uint64 beyond (n <= 2^40); a slice     */
/* holds at most HKCSA_MAX_N suffixes.  "peer" arrays: h_peer_x[r] is the device address, as mapped into THIS      */
/* process, of rank r's buffer x (torch symmetric memory / cudaIpc; plain local buffers when ranks are emulated).  */
#define HKCSA_DSA_BUCKETS 65536u
#define HKCSA_DSA_MAX_RANKS 8
#define HKCSA_DSA_MAX_N32 ((uint64_t)0xFFFFFFFEull)

typedef struct hkcsa_dsa_plan {   /* derived from the byte histogram of the WHOLE text: identical on every rank */
    uint64_t n;
    uint32_t sigma;
    uint32_t bits0;               /* width of a round-0 key (multiple of 8)                                     */
    uint32_t k0;                  /* symbols every round-0 key is guaranteed to cover                            */
    uint32_t passes0;             /* radix passes of the round-0 sort                                            */
    uint32_t b_fixed;             /* bits of a fixed-width symbol code (extension rounds)                        */
    uint32_t wide;                /* 1: suffix ids are uint64                                                    */
    uint32_t code[257];           /* the order-preserving prefix code of round 0 ([256] = past the end)          */
    uint8_t  len[257];
    uint16_t fixed_code[256];     /* dense code + 1 per byte, 0 = byte does not occur                            */
} hkcsa_dsa_plan;
typedef struct hkcsa_dsa_state { uint64_t opaque[512]; } hkcsa_dsa_state;   /* host-side, owned by the caller   */

int hkcsa_dsa_plan_make(const uint64_t *h_byte_hist, uint64_t n, int force_wide, hkcsa_dsa_plan *h_plan);
/* d_hist[HKCSA_DSA_BUCKETS] (overwritten): suffixes of [begin, end) per bucket = top 16 bits of the round-0 key  */
int hkcsa_dsa_bucket_hist(const uint8_t *d_text, const hkcsa_dsa_plan *h_plan, uint64_t begin, uint64_t end,
                          uint64_t *d_hist, void *stream);
/* The same over every tile_stride-th tile of 2048 positions only: cut points from a sample (one global atomic per  */
/* suffix is what the exact histogram costs).  The exact sizes of the exchange regions then come from              */
/* hkcsa_dsa_dest_counts: d_counts[HKCSA_DSA_MAX_RANKS] (overwritten) = suffixes of [begin, end) per owner rank.    */
int hkcsa_dsa_bucket_hist_sampled(const uint8_t *d_text, const hkcsa_dsa_plan *h_plan, uint64_t begin, uint64_t end,
                                  uint32_t tile_stride, uint64_t *d_hist, void *stream);
int hkcsa_dsa_dest_counts(const uint8_t *d_text, const hkcsa_dsa_plan *h_plan, uint64_t begin, uint64_t end,
                          uint32_t world, const uint32_t *h_cuts, uint64_t *d_counts, void *stream);
/* Pack + partition + exchange of the suffixes of [begin, end): rank r owns buckets [h_cuts[r], h_cuts[r+1]);     */
/* (key, id) pairs go to h_peer_keys[r] (uint64) / h_peer_ids[r] (uint32, or uint64 when plan->wide) from slot     */
/* h_base[r] on (this source's region; the caller sizes the regions from the all-gathered bucket histograms).      */
/* d_counters: uint64[HKCSA_DSA_MAX_RANKS], zeroed here, receives the pairs sent per destination.                  */
int hkcsa_dsa_pack_exchange(const uint8_t *d_text, const hkcsa_dsa_plan *h_plan, uint64_t begin, uint64_t end,
                            uint32_t world, const uint32_t *h_cuts, const uint64_t *h_peer_keys,
                            const uint64_t *h_peer_ids, const uint64_t *h_base, uint64_t *d_counters, void *stream);
/* Sort + refine the M received pairs.  d_keys: the received keys.  Narrow ids: d_ids == d_val_a = the received    */
/* uint32 ids; wide: d_ids = the received uint64 ids (kept intact), d_val_a a uint32[capacity] buffer.  d_val_b:    */
/* uint32[capacity].  The sorted slice (ids, or ordinals into d_ids when wide) ends up in d_val_a or d_val_b:      */
/* hkcsa_dsa_slice() tells which.  `capacity` must be the same on every rank.  Every call below syncs.             */
size_t hkcsa_dsa_state_bytes(void);
size_t hkcsa_dsa_scratch_bytes(uint64_t capacity);
int hkcsa_dsa_begin(hkcsa_dsa_state *state, const hkcsa_dsa_plan *h_plan, const uint8_t *d_text, uint64_t *d_keys,
                    void *d_ids, uint32_t *d_val_a, uint32_t *d_val_b, uint64_t M, uint64_t capacity,
                    void *d_scratch, size_t scratch_bytes, void *stream);
uint64_t hkcsa_dsa_working_set(const hkcsa_dsa_state *state);   /* suffixes in groups that are not singletons yet  */
uint64_t hkcsa_dsa_depth(const hkcsa_dsa_state *state);         /* symbols every group is known to share           */
const void *hkcsa_dsa_slice(const hkcsa_dsa_state *state);
int hkcsa_dsa_rounds(const hkcsa_dsa_state *state, uint32_t *h_rounds, uint64_t *h_round_elems, uint32_t max_rounds);
/* one round without a radix sort (local): groups of up to 16 suffixes are ordered by comparing the replicated text  */
/* beyond the current depth (up to 64 symbols); the depth does not advance.  Meant for the first round after _begin. */
int hkcsa_dsa_group_round(hkcsa_dsa_state *state, void *stream);
/* one extension round (local): the same number of symbols on every rank */
int hkcsa_dsa_ext_round(hkcsa_dsa_state *state, void *stream);
/* Rank doubling.  ISA blocks: rank r holds the global ranks of positions [r*blk, (r+1)*blk) as uint32 (uint64 when */
/* wide), all-ones = no entry; the caller fills them with 0xFF before the first publish.  A round is                */
/*   hkcsa_dsa_dbl_keys (reads peers) | ranks synchronise | hkcsa_dsa_dbl_sort (local) + hkcsa_dsa_isa_publish      */
/*   (writes peers, with_singles = 1) | ranks synchronise.                                                         */
/* The first publish (with_singles = 0) enters the working set as it stands after the extension rounds.            */
int hkcsa_dsa_isa_publish(hkcsa_dsa_state *state, uint32_t world, const uint64_t *h_peer_isa, uint64_t blk,
                          uint64_t slice_offset, int with_singles, void *stream);
int hkcsa_dsa_dbl_keys(hkcsa_dsa_state *state, uint32_t world, const uint64_t *h_peer_isa, uint64_t blk,
                       const uint64_t *h_peer_sa, const uint64_t *h_peer_ids64, const uint64_t *h_slice_off,
                       const uint32_t *h_cuts, void *stream);
int hkcsa_dsa_dbl_sort(hkcsa_dsa_state *state, void *stream);
/* wide ids: d_out[j] = id of the j-th suffix of the finished slice (uint64[M]); d_out_bwt (may be NULL) receives the  */
/* BWT slice: with 64-bit ids the exchange carries text[i-1] in the top byte of every id (n <= 2^40 leaves it free), */
/* so the slice's BWT costs no gather over the text                                                                   */
/* Layout of a 64-bit id word in the receive arrays: bits 0-39 suffix id, bits 40-55 the 16 bits of the round-0    */
/* code stream that follow the key (compared by the group round before it reads any text; 0 when a code word of one  */
/* bit makes them unavailable), bits 56-63 text[i-1].                                                                 */
int hkcsa_dsa_gather_ids64(const hkcsa_dsa_state *state, uint64_t *d_out, uint8_t *d_out_bwt, void *stream);
/* bwt[j] = text[SA[j]-1] (text[n-1] when SA[j] == 0) for a slice of the suffix array */
int hkcsa_bwt_slice(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa_slice, uint64_t m,
                    uint8_t *d_out, void *stream);
int hkcsa_bwt_slice64(const uint8_t *d_text, uint64_t n, const uint64_t *d_sa_slice, uint64_t m,
                      uint8_t *d_out, void *stream);

/* ------------------------------------------------------------------------ */
/* K2  BWT gather -- replaces bwt_transform, csa/bwt.py:3-13:                   */
/*     bwt[i] = text[SA[i]-1], text[n-1] when SA[i] == 0.                       */
/* ------------------------------------------------------------------------ */
int hkcsa_bwt(const uint8_t *d_text, const uint32_t *d_sa, uint64_t n, uint8_t *d_bwt, void *stream);

/* K1 + K2 in one call -- the pair EnhancedFMIndex.__init__ runs back to back,   */
/* csa/enhanced_fm_index.py:10-11 (build_suffix_array, then bwt_transform).       */
/* Same contract as hkcsa_sa_build plus d_bwt: uint8[n].  When the round-0 key    */
/* leaves its top byte free (<= 56 sorted bits) the symbol before each suffix     */
/* rides through the radix sort in that byte and the BWT is written while the     */
/* sorted keys are read -- no random gather over the text; otherwise the gather   */
/* of hkcsa_bwt runs after the build.  Identical outputs either way.  syncs.      */
int hkcsa_sa_bwt_build(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint8_t *d_bwt,
                       void *d_scratch, size_t scratch_bytes, void *stream, hkcsa_sa_stats *h_stats);

/* Byte histogram: the raw counts under build_count, utils/utils.py:16-24.      */
/* d_hist: uint64[256] (overwritten).                                           */
int hkcsa_byte_hist(const uint8_t *d_sym, uint64_t n, uint64_t *d_hist, void *stream);

/* ------------------------------------------------------------------------ */
/* K3  wavelet tree -- replaces WaveletTree.build_tree (csa/wavelet_tree.py:    */
/*     72-100), SuccinctRankSelect.__init__ (:6-12), build_count and build_occ  */
/*     (utils/utils.py:16-32).  Full level-wise tree with the reference's       */
/*     alphabet-halving split (mid = lo + (hi-lo)/2 over the sorted alphabet);  */
/*     the reference's levels are the first node of each level.                 */
/*                                                                              */
/*     Level bit-vectors are stored as 32-byte rank blocks (one DRAM sector):   */
/*       word0 low 32 bits  = ones before this block, relative to its superblock*/
/*       remaining 224 bits = payload, bit j of the level at (j % 224) + 32     */
/*     read as four little-endian uint64.  Superblocks (every 2^16 blocks) hold */
/*     absolute uint64 counts.  Select samples: position of every 4096-th one.  */
/* ------------------------------------------------------------------------ */
#define HKCSA_BLOCK_BITS 224u
#define HKCSA_SUPER_BLOCKS 65536u
#define HKCSA_SELECT_SAMPLE 4096u

typedef struct hkcsa_wt_plan {
    uint64_t n;                           /* symbols in the sequence (BWT)      */
    uint32_t sigma;                       /* distinct symbols                   */
    uint32_t levels;                      /* tree height (0 when sigma <= 1)    */
    uint8_t  sym_of_code[256];            /* dense code -> byte (sorted bytes)  */
    uint16_t code_of_sym[256];            /* byte -> dense code, 0xFFFF absent  */
    uint64_t cnt[256];                    /* occurrences per dense code         */
    uint64_t C[257];                      /* C[code] = symbols with smaller code*/
    uint8_t  depth[256];                  /* levels a code takes part in        */
    uint64_t level_len[HKCSA_MAX_LEVELS]; /* bits in each level                 */
    uint32_t level_nodes[HKCSA_MAX_LEVELS];
    /* byte offsets into the index blob */
    uint64_t off_tables;                  /* device copy of node tables         */
    uint64_t off_blocks[HKCSA_MAX_LEVELS];/* rank blocks of level l             */
    uint64_t off_super[HKCSA_MAX_LEVELS]; /* uint64 superblock counts           */
    uint64_t off_select[HKCSA_MAX_LEVELS];/* uint32 select samples              */
    uint64_t level_ones[HKCSA_MAX_LEVELS];/* filled by hkcsa_wt_build           */
    uint64_t blob_bytes;                  /* total size of the index blob       */
    uint64_t scratch_bytes;               /* scratch for hkcsa_wt_build         */
    /* per (level, code): node start in the level, the bit the code takes,      */
    /* the node id among the level's internal nodes (0xFF = not present)        */
    uint32_t node_start[HKCSA_MAX_LEVELS][256];
    uint8_t  node_bit[HKCSA_MAX_LEVELS][256];
    uint8_t  node_id[HKCSA_MAX_LEVELS][256];
} hkcsa_wt_plan;

/* Host-only: derive the tree shape and blob layout from a byte histogram.      */
int hkcsa_wt_plan_from_hist(const uint64_t h_hist[256], hkcsa_wt_plan *h_plan);
/* Builds every level, its rank blocks, superblocks and select samples into     */
/* d_blob (plan->blob_bytes, 32-byte aligned).  syncs once at the end to fill   */
/* plan->level_ones.  d_sym: the sequence as raw bytes (the BWT).               */
int hkcsa_wt_build(const uint8_t *d_sym, hkcsa_wt_plan *h_plan, void *d_blob, void *d_scratch,
                   size_t scratch_bytes, void *stream);

/* Bit-vector primitives on one level -- SuccinctRankSelect.rank/select,        */
/* csa/wavelet_tree.py:14-25.  rank(i) = ones in bits[0:i], i in [0, len];      */
/* select(k) = smallest p in [0,len] with rank(p) >= k.                         */
int hkcsa_bv_rank_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                        const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream);
int hkcsa_bv_select_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                          const uint64_t *d_k, uint64_t m, uint64_t *d_out, void *stream);
/* Unpack bits [begin, begin+count) of a level to one byte per bit (the          */
/* SuccinctRankSelect.bit_vector view, csa/wavelet_tree.py:8).                  */
int hkcsa_bv_unpack(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                    uint64_t begin, uint64_t count, uint8_t *d_out, void *stream);
/* rank_support[begin .. begin+count) as uint32 (csa/wavelet_tree.py:9-12).     */
int hkcsa_bv_rank_range(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                        uint64_t begin, uint64_t count, uint32_t *d_out, void *stream);

/* Stand-alone bit-vector: SuccinctRankSelect(bitmap) outside a tree              */
/* (csa/wavelet_tree.py:5-25).  hkcsa_bitvec_plan fills a one-level plan whose    */
/* level 0 is the bitmap, so the hkcsa_bv_* queries apply with level = 0.         */
/* d_bits: one byte per bit (non-zero = 1).  hkcsa_bitvec_build syncs.            */
int hkcsa_bitvec_plan(uint64_t nbits, hkcsa_wt_plan *h_plan);
int hkcsa_bitvec_build(const uint8_t *d_bits, hkcsa_wt_plan *h_plan, void *d_blob, void *d_scratch,
                       size_t scratch_bytes, void *stream);

/* Stable bucket partition of a byte sequence by a host byte -> bucket table      */
/* (bucket 255 sorts last: use it for "drop").  next_text of the reference        */
/* (csa/wavelet_tree.py:92) is bucket 0 of {left alphabet -> 0, rest -> 255}.     */
/* h_bucket_sizes: uint64[256] out.  syncs.                                       */
size_t hkcsa_partition_scratch_bytes(uint64_t n);
int hkcsa_partition_bytes(const uint8_t *d_in, uint64_t n, const uint8_t *h_lut, uint8_t *d_out,
                          uint64_t *h_bucket_sizes, void *d_scratch, size_t scratch_bytes, void *stream);

/* Symbol-level queries: occ[c][i] of build_occ (utils/utils.py:26-32) ==       */
/* EnhancedFMIndex.rank (csa/enhanced_fm_index.py:34-40), and access (bwt[i]).  */
/* d_sym: query bytes; a byte that never occurs answers 0.                      */
int hkcsa_wt_rank_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint8_t *d_sym,
                        const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream);
int hkcsa_wt_access_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint64_t *d_pos,
                          uint64_t m, uint8_t *d_out, void *stream);

/* Golomb-Rice run code of a level's first node (the reference's                */
/* tree[l][0]) -- GolombRiceEncoder, csa/wavelet_tree.py:27-63.                 */
/* Encodes bits [0, nbits) of `level`; m as computed by :33-38.  Two calls:     */
/* d_out == NULL sizes the output (*h_out_bits), otherwise writes one byte per  */
/* code bit.  syncs.                                                            */
int hkcsa_golomb_encode(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t level,
                        uint64_t nbits, uint32_t m, uint8_t *d_out, uint64_t out_capacity,
                        uint64_t *h_out_bits, void *d_scratch, size_t scratch_bytes, void *stream);
size_t hkcsa_golomb_scratch_bytes(uint64_t nbits);

/* ------------------------------------------------------------------------ */
/* K4  FM backward search -- replaces EnhancedFMIndex.find_range / .rank /      */
/*     .find, csa/enhanced_fm_index.py:15-40.                                   */
/*     Patterns: concatenated bytes + int64 offsets[P+1].                       */
/*     count: inclusive SA range (lo, hi); miss = (-1, -1); empty pattern =     */
/*     (0, n-1).  Same recurrences and miss conventions as :21-32.              */
/* ------------------------------------------------------------------------ */
int hkcsa_count_batch(const void *d_blob, const hkcsa_wt_plan *h_plan, const uint8_t *d_pat,
                      const int64_t *d_off, uint64_t P, int64_t *d_lo, int64_t *d_hi, void *stream);

/* k-mer jump table: the SA range of every k-mer over the index alphabet (k = hkcsa_kmer_k(sigma): the   */
/* largest k with sigma^k <= 2^21), computed by the count kernel itself.  hkcsa_count_batch_kmer starts   */
/* every pattern of length >= k from the table entry of its last k symbols and continues backwards: the   */
/* results are identical to hkcsa_count_batch, k rank steps cheaper.  d_table: 8 bytes per entry.         */
uint32_t hkcsa_kmer_k(uint32_t sigma);
uint64_t hkcsa_kmer_entries(uint32_t sigma, uint32_t k);
size_t hkcsa_kmer_scratch_bytes(uint32_t sigma, uint32_t k);
int hkcsa_kmer_table_build(const void *d_blob, const hkcsa_wt_plan *h_plan, uint32_t k, void *d_table,
                           void *d_scratch, size_t scratch_bytes, void *stream);
int hkcsa_count_batch_kmer(const void *d_blob, const hkcsa_wt_plan *h_plan, const void *d_kmer_table, uint32_t k,
                           const uint8_t *d_pat, const int64_t *d_off, uint64_t P, int64_t *d_lo, int64_t *d_hi,
                           void *stream);

/* Sampled suffix array for locate: marks rows with SA[j] % rate == 0 (a rank   */
/* bit-vector in the block format above) and stores SA[j] / rate for them.      */
typedef struct hkcsa_ssa_plan {
    uint64_t n;
    uint32_t rate;
    uint64_t n_samples;      /* ceil(n / rate)                                  */
    uint64_t off_blocks;     /* mark bit-vector rank blocks                     */
    uint64_t off_super;
    uint64_t off_samples;    /* uint32[n_samples]                               */
    uint64_t blob_bytes;
    uint64_t scratch_bytes;
} hkcsa_ssa_plan;

int hkcsa_ssa_plan_make(uint64_t n, uint32_t rate, hkcsa_ssa_plan *h_plan);
int hkcsa_ssa_build(const uint32_t *d_sa, const hkcsa_ssa_plan *h_plan, void *d_blob, void *d_scratch,
                    size_t scratch_bytes, void *stream);

/* locate, step 1: expand SA ranges into rows.  d_out_off: int64[P+1] exclusive */
/* prefix sums of (hi-lo+1) (0 for misses), computed by the caller.             */
int hkcsa_expand_ranges(const int64_t *d_lo, const int64_t *d_hi, const int64_t *d_out_off, uint64_t P,
                        uint32_t *d_rows, void *stream);
/* locate, step 2a: positions from the full SA (what EnhancedFMIndex.find does,  */
/* csa/enhanced_fm_index.py:19): out[q] = SA[rows[q]], SA order preserved.       */
int hkcsa_gather_u32(const uint32_t *d_src, const uint32_t *d_rows, uint64_t m, uint32_t *d_out,
                     void *stream);
/* locate, step 2b: positions by LF walk to the next sampled row.  row0 = the   */
/* row of suffix 0 (hkcsa_isa_samples()[0]).  The LF step is exact on every text */
/* (also one that holds its last symbol elsewhere, e.g. a second '$': occ alone  */
/* would misrank row0 there), so a walk meets a marked row within rate-1 steps; */
/* a walk that exceeds them (only on a corrupt index) stops and writes          */
/* HKCSA_NO_POSITION instead of spinning.                                        */
#define HKCSA_NO_POSITION 0xFFFFFFFFu
int hkcsa_locate_rows(const void *d_wt_blob, const hkcsa_wt_plan *h_plan, const void *d_ssa_blob,
                      const hkcsa_ssa_plan *h_ssa, uint32_t row0, const uint32_t *d_rows, uint64_t m,
                      uint32_t *d_out_pos, void *stream);

/* ------------------------------------------------------------------------ */
/* The constructor in one call -- EnhancedFMIndex.__init__,                    */
/* csa/enhanced_fm_index.py:8-13 (suffix array, BWT, occ / count): suffix array */
/* + BWT on `stream` (hkcsa_sa_bwt_build), then the wavelet tree over the BWT   */
/* on `stream_tree` and the sampled suffix array on `stream_ssa` side by side   */
/* (NULL = `stream`); on return `stream` waits for both.  h_ssa_plan NULL = no  */
/* sampled SA.  The tree's shape depends on the byte histogram, which the call  */
/* computes itself: the caller sizes d_wt_blob / d_wt_scratch with the bounds   */
/* below, the plan filled into h_wt_plan says how much of the blob is used.     */
/* No host-language code runs between the refinement rounds and the tree        */
/* kernels -- the GPU does not wait for the caller there.  syncs.               */
size_t hkcsa_wt_blob_bound(uint64_t n);
size_t hkcsa_wt_scratch_bound(uint64_t n);
int hkcsa_index_build(const uint8_t *d_text, uint64_t n, uint32_t *d_sa, uint8_t *d_bwt, void *d_sa_scratch,
                      size_t sa_scratch_bytes, hkcsa_wt_plan *h_wt_plan, void *d_wt_blob, size_t wt_blob_cap,
                      void *d_wt_scratch, size_t wt_scratch_cap, const hkcsa_ssa_plan *h_ssa_plan,
                      void *d_ssa_blob, void *d_ssa_scratch, size_t ssa_scratch_bytes, void *stream,
                      void *stream_tree, void *stream_ssa, hkcsa_sa_stats *h_stats);

/* Sampled SA of a SLICE of the suffix array (distributed build): the number of marked rows of a slice is  */
/* not ceil(m / rate), the caller passes it (count of SA[j] % rate == 0 in the slice).                        */
int hkcsa_ssa_plan_make_slice(uint64_t m, uint32_t rate, uint64_t n_marks, hkcsa_ssa_plan *h_plan);
/* hkcsa_ssa_build for uint64 suffix ids (samples stay uint32: id / rate must fit)                            */
int hkcsa_ssa_build64(const uint64_t *d_sa, const hkcsa_ssa_plan *h_plan, void *d_blob, void *d_scratch,
                      size_t scratch_bytes, void *stream);
int hkcsa_expand_ranges64(const int64_t *d_lo, const int64_t *d_hi, const int64_t *d_out_off, uint64_t P,
                          uint64_t *d_rows, void *stream);

/* Backward search over a BWT built in slices (BASELINE config 5): slice s covers global rows                 */
/* [h_starts[s], h_starts[s+1]) with its own wavelet-tree blob / plan (hkcsa_wt_build over its BWT slice) and, */
/* optionally, its own sampled SA.  The descriptor lives in device memory (hkcsa_multi_desc_bytes()).          */
/* Same recurrences and miss conventions as hkcsa_count_batch; rows and positions are global (n <= 2^40).      */
/* row0 = the global row of suffix 0 (< n), UINT64_MAX when there is no sampled SA: the LF step of locate is   */
/* the exact one of hkcsa_locate_rows, also on a text that holds its last symbol elsewhere.                    */
#define HKCSA_MAX_SLICES 8
size_t hkcsa_multi_desc_bytes(void);
int hkcsa_multi_desc_build(uint32_t S, const void *const *d_wt_blobs, const hkcsa_wt_plan *const *h_plans,
                           const uint64_t *h_starts, const void *const *d_ssa_blobs,
                           const hkcsa_ssa_plan *const *h_ssa_plans, uint64_t row0, void *d_desc, void *stream);
int hkcsa_multi_count_batch(const void *d_desc, const uint8_t *d_pat, const int64_t *d_off, uint64_t P,
                            int64_t *d_lo, int64_t *d_hi, void *stream);
/* rows and positions are 64-bit (the sliced index may exceed 2^32 rows): use hkcsa_expand_ranges64.  A walk  */
/* longer than rate steps (a corrupt index only) writes HKCSA_NO_POSITION64 (-1 as int64).                    */
#define HKCSA_NO_POSITION64 0xFFFFFFFFFFFFFFFFull
int hkcsa_multi_locate_rows(const void *d_desc, const uint64_t *d_rows, uint64_t m, uint64_t *d_out_pos,
                            void *stream);

/* FMIndex.precompute_rank, csa/csa.py:13-19: positions of every symbol in the  */
/* BWT, ascending, grouped by byte value (a stable counting sort).  d_start:    */
/* uint64[257].  d_scratch: hkcsa_symbol_positions_scratch_bytes(n).                      */
size_t hkcsa_symbol_positions_scratch_bytes(uint64_t n);
int hkcsa_symbol_positions(const uint8_t *d_bwt, uint64_t n, uint32_t *d_pos, uint64_t *d_start,
                           void *d_scratch, size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------ */
/* Entropy-coded bit-vectors with rank on the coded form (no working reference   */
/* counterpart: WaveletTree.compress keeps Golomb run codes that cannot be       */
/* decoded -- zero runs are not coded, csa/wavelet_tree.py:40-63 -- and          */
/* decompress returns '', :158-200).  Class/offset code of Raman-Raman-Rao with   */
/* 15-bit blocks: per block a 4-bit class (its popcount) and the index of the     */
/* pattern inside its class in ceil(log2 C(15, c)) bits; per 64 blocks the ones   */
/* and the offset-stream position before them (2 x 32 bits).  n H_0 + o(n) bits per vector;     */
/* over the wavelet-tree levels of a BWT that is the n H_k + o(n) index.          */
/* ------------------------------------------------------------------------ */
typedef struct hkcsa_rrr_plan {
    uint64_t nbits, nblocks, nsuper;
    uint64_t ones;           /* ones in the vector                               */
    uint64_t stream_bits;    /* length of the offset stream                      */
    uint64_t off_super, off_classes, off_stream;
    uint64_t blob_bytes;
} hkcsa_rrr_plan;
size_t hkcsa_rrr_tables_bytes(void);
int hkcsa_rrr_tables_init(void *d_tables, void *stream);              /* syncs */
size_t hkcsa_rrr_scratch_bytes(uint64_t nbits);
/* Encodes bits [0, nbits) of `level` of a wavelet-tree blob.  Two calls: d_out == NULL sizes the code (fills   */
/* *h_plan), otherwise writes it (h_plan->blob_bytes bytes, 32-byte aligned, out_capacity >= that).  syncs.      */
int hkcsa_rrr_encode(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, uint32_t level, uint64_t nbits,
                     const void *d_tables, hkcsa_rrr_plan *h_plan, void *d_out, size_t out_capacity,
                     void *d_scratch, size_t scratch_bytes, void *stream);
/* SuccinctRankSelect.rank (csa/wavelet_tree.py:14-15) on the coded form: ones in bits [0, i) */
int hkcsa_rrr_rank_batch(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables,
                         const uint64_t *d_pos, uint64_t m, uint64_t *d_out, void *stream);
/* bits [begin, begin + count) decoded to one byte per bit */
int hkcsa_rrr_unpack(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables, uint64_t begin,
                     uint64_t count, uint8_t *d_out, void *stream);
/* Restoring a wavelet-tree blob from coded levels: hkcsa_wt_restore_begin writes the node tables and clears the  */
/* level regions, hkcsa_rrr_restore_level decodes a level's payload bits in place, hkcsa_wt_restore_finish        */
/* rebuilds block headers, superblocks, select samples and node counts (scratch: plan->scratch_bytes) and checks  */
/* the ones per level against the plan.                                                                           */
int hkcsa_wt_restore_begin(const hkcsa_wt_plan *h_plan, void *d_blob, void *stream);
int hkcsa_rrr_restore_level(const void *d_rrr, const hkcsa_rrr_plan *h_plan, const void *d_tables,
                            const hkcsa_wt_plan *h_wt_plan, uint32_t level, void *d_wt_blob, void *stream);
int hkcsa_wt_restore_finish(const hkcsa_wt_plan *h_plan, void *d_blob, void *d_scratch, size_t scratch_bytes,
                            void *stream);

/* ------------------------------------------------------------------------ */
/* k-th order empirical entropy -- replaces calculate_high_order_entropy,       */
/* csa/high_order_entropy.py:4-32, for k >= 1 (H_0 follows from hkcsa_byte_hist).*/
/* The windows text[i : i+k+1] sharing a (k+1)-gram are a run of adjacent        */
/* suffixes, so the suffix array of the text gives H_k for ANY k in one pass:    */
/*   h_out[0] = sum over k-gram contexts of T log2 T, h_out[1] = sum over        */
/*   (k+1)-grams of c log2 c, h_out[2] = windows (n - k), h_out[3] / h_out[4] =  */
/*   distinct contexts / (k+1)-grams;  H_k = (h_out[0] - h_out[1]) / n  (the     */
/*   reference divides by n, not n - k: :30).  fp64, fixed summation order.      */
/*   n <= k -> all zeros (:17-18).  syncs.                                       */
/* ------------------------------------------------------------------------ */
size_t hkcsa_entropy_scratch_bytes(uint64_t n);
int hkcsa_entropy_from_sa(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t k, double *h_out /* [5] */,
                          void *d_scratch, size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------ */
/* K6  LCP -- longest common prefixes of adjacent suffixes (no reference       */
/*     counterpart).  LCP[0] = 0, LCP[r] = lcp(text[SA[r-1]:], text[SA[r]:])   */
/*     (SA order); PLCP[i] = LCP[ISA[i]] (text order).  Any text, sentinel or  */
/*     not; values < n, stored as uint32.  Irreducible-PLCP method            */
/*     (Karkkainen-Manzini-Puglisi 2009): only positions i with i == 0,        */
/*     Phi[i] == 0, text[i-1] != text[Phi[i]-1] or i == SA[0] are compared     */
/*     (their values sum to <= 2 n log2 n), the rest by a max-scan.            */
/*     Scratch: 4n bytes (Phi with its flag, then PLCP) + 16 bytes per position */
/*     of a chunk of min(n, max(2^22, n/16)) positions (the lists of long      */
/*     pairs) -- about 5n bytes beside text, SA and outputs at HKCSA_MAX_N.    */
/* ------------------------------------------------------------------------ */
size_t hkcsa_lcp_scratch_bytes(uint64_t n);
/* LCP (SA order) and / or PLCP (text order) of any text from its suffix array; either output may be NULL (not both).
   h_stats: NULL, or uint64[2] = {irreducible positions, sum of their values} (then the call syncs; otherwise it does not). */
int hkcsa_lcp_build(const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint32_t *d_lcp, uint32_t *d_plcp,
                    void *d_scratch, size_t scratch_bytes, uint64_t *h_stats, void *stream);
/* Sadakane's encoding: d_bits[PLCP[i] + 2 i] = 1 for every i, all other bytes 0; d_bits holds 2n bytes (one per bit,
   the input format of hkcsa_bitvec_build).  Then PLCP[i] = select(i + 1) - 1 - 2 i. */
int hkcsa_plcp_bits(const uint32_t *d_plcp, uint64_t n, uint8_t *d_bits, void *stream);

/* ------------------------------------------------------------------------ */
/* Measurement hook (no reference counterpart; the reference times with       */
/* time.time(), tests/benchmark.py:30-35).  When enabled, the library brackets */
/* its own kernel launches with CUDA events on the launching stream;           */
/* hkcsa_prof_read syncs on them and returns one entry per kernel class.       */
/* ------------------------------------------------------------------------ */
typedef struct hkcsa_prof_entry {
    char     name[32];
    uint64_t launches;
    double   ms;          /* summed device time between the bracketing events  */
    uint64_t alg_bytes;   /* summed algorithmic bytes (DESIGN.md, per kernel)   */
} hkcsa_prof_entry;
#define HKCSA_PROF_CLASSES 16
/* kernels launched by the library so far in this process */
unsigned long long hkcsa_launch_count(void);
int hkcsa_prof_enable(int on);
/* time only the classes whose bit is set (bit = hkcsa_prof_class_index(name)): a timed region that needs one */
/* kernel's durations does not pay two event records around every other launch                                */
int hkcsa_prof_enable_classes(uint32_t class_mask);
int hkcsa_prof_class_index(const char *name);
int hkcsa_prof_reset(void);
int hkcsa_prof_read(hkcsa_prof_entry *h_out, int max_entries, int *h_n);
/* every bracketed launch in recording order: start / end (ms after the first record's start) and class index    */
int hkcsa_prof_timeline(float *h_start_ms, float *h_end_ms, int *h_class, int max_entries, int *h_n);

/* ------------------------------------------------------------------------ */
/* Sampled Occ table (optional second rank structure): the reference's dense occ[c][i] (build_occ,          */
/* utils/utils.py:26-32; read by EnhancedFMIndex.rank, csa/enhanced_fm_index.py:34-40) kept at every       */
/* 2^shift-th row, each kept row stored next to the 2^shift BWT bytes the remainder is counted from:       */
/*   row r = [2^shift BWT bytes][sigma x uint32 occ[code][r << shift]], `stride` bytes apart, rows = (n >> shift) + 1. */
/* One rank touches one counter sector + the symbol sector(s), whatever the alphabet (the wavelet tree: one */
/* sector per level).  hkcsa_count_batch_occ returns exactly what hkcsa_count_batch returns.                */
typedef struct hkcsa_occ_plan {
    uint64_t n;
    uint32_t sigma;
    uint32_t shift;          /* 5 or 6 */
    uint32_t layout;         /* 0: rows as above.  1 (shift 5): per symbol and per 32 rows ONE 8-byte entry         */
    uint32_t reserved;       /*    { occ[code][32 r], bitmap of the rows 32 r .. 32 r + 31 holding `code` }: a rank  */
                             /*    is one memory request; entry[code * stride + r]; the blob ends with a BWT copy   */
    uint64_t off_bwt;        /* layout 1: byte offset of the BWT copy (LF steps of locate)                          */
    uint64_t rows;
    uint64_t stride;         /* layout 0: bytes per row, multiple of 32; layout 1: entries per code */
    uint64_t blob_bytes;
    uint64_t scratch_bytes;  /* for hkcsa_occ_build */
} hkcsa_occ_plan;
int hkcsa_occ_plan_make(uint64_t n, uint32_t sigma, uint32_t shift, uint32_t layout, hkcsa_occ_plan *h_plan);
int hkcsa_occ_build(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const uint8_t *d_bwt,
                    const hkcsa_occ_plan *h_plan, void *d_blob, void *d_scratch, size_t scratch_bytes, void *stream);
int hkcsa_count_batch_occ(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const void *d_occ_blob,
                          const hkcsa_occ_plan *h_plan, const void *d_kmer_table, uint32_t k, const uint8_t *d_pat,
                          const int64_t *d_off, uint64_t P, int64_t *d_lo, int64_t *d_hi, void *stream);
/* Multi-GPU count with the gather of the results fused into the search: this rank's kernel writes the ranges of */
/* its P patterns (a slice of the global batch starting at out_base) into the lo / hi arrays of ALL n_peers ranks  */
/* through peer-mapped device pointers (h_peer_lo[r], h_peer_hi[r]: int64 arrays of the global batch size, e.g.    */
/* torch symmetric memory or cudaIpc mappings; the own rank included).  No collective follows; the caller        */
/* synchronises the ranks before reading.  d_occ_blob / h_occ_plan may both be NULL (wavelet-tree ranks).          */
#define HKCSA_MAX_PEERS 16
int hkcsa_count_batch_peers(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const void *d_occ_blob,
                            const hkcsa_occ_plan *h_occ_plan, const void *d_kmer_table, uint32_t k,
                            const uint8_t *d_pat, const int64_t *d_off, uint64_t P, uint64_t out_base,
                            uint32_t n_peers, const uint64_t *h_peer_lo, const uint64_t *h_peer_hi, void *stream);
/* The gather of a sharded batch's results as a store kernel: (lo, hi) of this rank's P patterns are packed into     */
/* 8 bytes {lo: low 32 bits, count = hi-lo+1: high 32 bits; miss: lo = 0xFFFFFFFF, count 0} and stored at             */
/* [out_base + p] of the uint64 result array of every rank (h_peer_out[r], peer-mapped, 16-byte aligned) -- or, when  */
/* multicast_out != 0 (the NVSwitch multicast address of the same symmetric array), by ONE multimem.st per 16 bytes   */
/* that reaches all ranks.  hkcsa_ranges_unpack expands a packed array back to (lo, hi).                              */
int hkcsa_ranges_push_peers(const int64_t *d_lo, const int64_t *d_hi, uint64_t P, uint64_t out_base,
                            uint32_t n_peers, const uint64_t *h_peer_out, uint64_t multicast_out, void *stream);
int hkcsa_ranges_unpack(const uint64_t *d_packed, uint64_t P, int64_t *d_lo, int64_t *d_hi, void *stream);
/* hkcsa_locate_rows with the LF step (symbol + its count) read from the Occ table; same positions. */
int hkcsa_locate_rows_occ(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const void *d_occ_blob,
                          const hkcsa_occ_plan *h_plan, const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa,
                          uint32_t row0, const uint32_t *d_rows, uint64_t m, uint32_t *d_out_pos, void *stream);

/* ------------------------------------------------------------------------ */
/* K4c extract: text[begin:end) back out of the index, without the text (no  */
/* reference counterpart: WaveletTree.decompress returns '',                  */
/* csa/wavelet_tree.py:158-200).                                              */
/* hkcsa_isa_samples: isa[k] = row of the suffix at text position k * rate    */
/* for k < S = h_ssa->n_samples, and isa[S] = isa[0]; derived from the        */
/* sampled SA alone (works on a loaded index).  A slice plan                  */
/* (hkcsa_ssa_plan_make_slice) is refused.  d_isa: uint32[S + 1].             */
/* hkcsa_extract: R requests [d_begin[q], d_end[q]) over the indexed text     */
/* (sentinel included), 0 <= begin <= end <= n; the bytes of request q go to  */
/* d_out[d_out_off[q] .. d_out_off[q+1]) (the caller's exclusive prefix sum   */
/* of end - begin).  Ranges are clamped on the device, so a bad one never     */
/* writes outside its own slice.  Each request runs as one LF walk per        */
/* sample block it touches, <= rate steps each.  d_occ_blob / h_occ_plan both */
/* NULL: LF on the wavelet tree; otherwise on the sampled Occ table (layout 0 */
/* or 1).  LF inverts the suffix order only when the text's sentinel is       */
/* unique (more precisely: when occ(bwt[isa[0]], isa[0]) == 0); on any other  */
/* index the bytes are not the text.                                          */
/* ------------------------------------------------------------------------ */
int    hkcsa_isa_samples(const void *d_ssa_blob, const hkcsa_ssa_plan *h_ssa, uint32_t *d_isa, void *stream);
size_t hkcsa_extract_scratch_bytes(uint64_t R);
int    hkcsa_extract(const void *d_wt_blob, const hkcsa_wt_plan *h_wt_plan, const void *d_occ_blob,
                     const hkcsa_occ_plan *h_occ_plan, const uint32_t *d_isa, uint32_t rate, const int64_t *d_begin,
                     const int64_t *d_end, const int64_t *d_out_off, uint64_t R, uint8_t *d_out, void *d_scratch,
                     size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------ */
/* K4c over the sliced index of the distributed build (hkcsa_multi_*).       */
/* hkcsa_multi_isa_samples: the same isa[] as hkcsa_isa_samples, as global   */
/* 64-bit rows, from the S slices' sampled SAs (h_starts as for              */
/* hkcsa_multi_desc_build).  Checked on the host before any CUDA call: equal */
/* rates, each plan's n == its slice length, the slices' n_samples add up to */
/* ceil(n / rate) (slices of one build), ceil(n / rate) <= 2^32 (samples are */
/* 32-bit), n <= 2^40.  d_isa: uint64[ceil(n / rate) + 1].                   */
/* hkcsa_multi_extract: hkcsa_extract's contract (CSR output, ranges clamped */
/* on the device, scratch from hkcsa_extract_scratch_bytes(R)) over the      */
/* descriptor of hkcsa_multi_desc_build, which must carry the sampled SAs    */
/* and row0; n and rate are the index's.  The LF step is the exact one of    */
/* hkcsa_multi_locate_rows, so the bytes are the text on every text, also    */
/* one that holds its last symbol elsewhere.                                 */
/* ------------------------------------------------------------------------ */
int hkcsa_multi_isa_samples(uint32_t S, const void *const *d_ssa_blobs, const hkcsa_ssa_plan *const *h_ssa_plans,
                            const uint64_t *h_starts, uint64_t *d_isa, void *stream);
int hkcsa_multi_extract(const void *d_desc, uint64_t n, uint32_t rate, const uint64_t *d_isa, const int64_t *d_begin,
                        const int64_t *d_end, const int64_t *d_out_off, uint64_t R, uint8_t *d_out, void *d_scratch,
                        size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------ */
/* Host text in, index out: the reference's constructor takes a Python str   */
/* (EnhancedFMIndex.__init__, csa/enhanced_fm_index.py:8-9; the corpus loader */
/* returns one, utils/data_loader.py:4) whose bytes sit in PAGEABLE memory.   */
/* hkcsa_h2d_staged copies nbytes from pageable h_src to d_dst through a      */
/* library-owned pinned ring (64 MB, allocated on first use): `threads` host  */
/* threads (0 = HKCSA_STAGE_THREADS or 4; at most 16) fill 2 MB               */
/* slots and enqueue each slot's DMA on `stream` as soon as it is filled, so  */
/* the host copy runs on several cores and overlaps the PCIe transfer.        */
/* Returns when every byte has been staged (h_src may be released); the DMAs  */
/* complete in stream order.  hkcsa_d2h_staged is the way back (index blobs,  */
/* suffix array): returns when h_dst holds the data.                          */
/* ------------------------------------------------------------------------ */
int hkcsa_h2d_staged(void *d_dst, const void *h_src, size_t nbytes, int threads, void *stream);
int hkcsa_d2h_staged(void *h_dst, const void *d_src, size_t nbytes, int threads, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HKCSA_H */
