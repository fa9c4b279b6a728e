"""The succinct primitives under the index, checked against exact references at every density and chunk boundary up to
the single-GPU limit of 2^30 - 2 bits:

* the stand-alone bit-vector (DeviceBitVector: hkcsa_bitvec_build + hkcsa_bv_*, csrc/wavelet.cu), which the drop-in
  SuccinctRankSelect and the LCP encoding use: ones, unpack, rank at every block and superblock edge, rank_range across
  a superblock, select at every select sample and its neighbours, on empty, full, single-one, sparse, dense, exact
  multiples of 4096 ones, ones in the last superblock only, and raw bytes where any nonzero byte is a one;
* the RRR class / offset code (RrrVector, csrc/rrr.cu): the plan's size fields, decode, and rank on the coded form past
  the 1024 superblocks one iteration of the single-CTA scan covers; every 15-bit pattern; coded wavelet-tree levels
  restored into a bit-identical query blob; a level prefix that ends inside a block;
* the Golomb run code (hkcsa_golomb_encode, csrc/golomb.cu): runs carried across a warp of 1792-bit chunks and across
  the 1024-chunk iterations of the single-CTA carry scan, runs closed by the end of input, every m up to 62, and level
  prefixes that end inside a run.

References: tests/succinct_reference.py and device_reference.bits_rank / bits_select on the device, the CPU oracle where
the vector has at most ~10^7 bits.  Every input comes from a seeded device generator.  A case skips only when the
device has less free memory than it needs (the number is in the reason).  The argument checks that need no device run
without the gpu mark."""
import ctypes as C

import numpy as np
import pytest
import torch

import device_reference as R
import succinct_reference as S
from hkcsa import _lib
from oracle import oracle as O

gpu = pytest.mark.gpu

# Geometry of the kernels under test -- keep in step with the sources named.
BLOCK_BITS = 224                     # payload bits of a rank block (hkcsa.h:225)
SUPER_BLOCKS = 65536                 # rank blocks per superblock (hkcsa.h:226)
SELECT_SAMPLE = 4096                 # ones per select sample (hkcsa.h:227)
SUPER_BITS = BLOCK_BITS * SUPER_BLOCKS
PACK_TILE_BITS = 14336               # bits per CTA of wt_pack_kernel (wavelet.cu:19-20)
RRR_B, RRR_SB = 15, 64               # bits per block, blocks per superblock of the class / offset code (rrr.cu:22-23)
RRR_SB_BITS = 960                    # (rrr.cu:24)
GOLOMB_CHUNK = 1792                  # bits per thread of the Golomb kernels (golomb.cu:17-19)
SCAN = 1024                          # elements per iteration of the single-CTA scans (golomb.cu:68, rrr.cu:111)
WARP = 32

MAX_N = _lib.MAX_N                   # 2^30 - 2
GB = 1 << 30
ORACLE_MAX = 10_000_000              # the CPU oracle checks vectors up to this many bits as well
UNPACK_CHUNK = 1 << 26


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _need_memory(dev, need, what):
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need:
        pytest.skip(f"{what}: needs {need / GB:.1f} GiB of device memory, {free / GB:.1f} GiB free")


def _assert_same(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    if torch.equal(got, want):
        return
    bad = (got != want).nonzero().flatten()
    i = int(bad[0])
    lo, hi = max(0, i - 2), min(got.numel(), i + 3)
    raise AssertionError(f"{what}: {bad.numel()} of {got.numel()} entries differ, first at {i}: "
                         f"got {got[lo:hi].tolist()}, want {want[lo:hi].tolist()} (entries {lo}..{hi - 1})")


def _bernoulli(n, p, g, dev, out=None, chunk=1 << 26):
    out = torch.empty(n, dtype=torch.uint8, device=dev) if out is None else out
    for a, b in R._chunks(n, chunk):
        out[a:b] = torch.rand(b - a, generator=g, device=dev) < p
    return out


def _i64(values, dev):
    return torch.as_tensor(values, dtype=torch.int64, device=dev)


# ------------------------------------------------------------------ bit-vector contents
def _bv_input(kind, n, seed, dev):
    """uint8[n] on the device; every kind but "bytes" holds 0 / 1."""
    g = torch.Generator(device=dev).manual_seed(seed)
    bits = torch.zeros(n, dtype=torch.uint8, device=dev)
    if n == 0 or kind == "zeros":
        return bits
    if kind == "ones":
        bits.fill_(1)
    elif kind == "first":
        bits[0] = 1
    elif kind == "last":
        bits[n - 1] = 1
    elif kind.startswith("p="):
        _bernoulli(n, {"p=1e-6": 1e-6, "p=0.5": 0.5, "p=1-1e-6": 1 - 1e-6}[kind], g, dev, out=bits)
    elif kind == "ones_4096j":             # exactly 4096 j ones: the last select sample's successor is the end
        j = min(n // SELECT_SAMPLE, 256)
        bits[torch.randperm(n, generator=g, device=dev)[:SELECT_SAMPLE * j]] = 1
    elif kind == "last_super":             # sparse ones from the last full superblock on, and bit n - 1: every
        start = max(0, n // SUPER_BITS - 1) * SUPER_BITS     # earlier superblock count is 0, samples are far apart
        _bernoulli(n - start, 1e-3, g, dev, out=bits[start:])
        bits[n - 1] = 1
    elif kind == "bytes":                  # any nonzero byte is a one (wavelet.cu:1147)
        bits = torch.randint(0, 256, (n,), dtype=torch.uint8, generator=g, device=dev)
    else:
        raise ValueError(kind)
    return bits


BV_LENGTHS = [0, 1, 223, 224, 225, PACK_TILE_BITS - 1, PACK_TILE_BITS, PACK_TILE_BITS + 1,
              SUPER_BITS - 1, SUPER_BITS, SUPER_BITS + 1, 3 * SUPER_BITS + 5]
BV_KINDS = ["zeros", "ones", "first", "last", "p=1e-6", "p=0.5", "p=1-1e-6", "ones_4096j", "last_super", "bytes"]
BV_MAX_KINDS = ["zeros", "ones", "p=1e-6", "p=0.5", "last_super"]
BV_CASES = [(n, k) for n in BV_LENGTHS for k in BV_KINDS] + [(MAX_N, k) for k in BV_MAX_KINDS]


def _rank_positions(n, g, dev):
    """0, n, n + 7 (clamped by the kernel), every rank-block edge +-1 of one full superblock (the last one, or the
    only one), every superblock edge +-1, and random positions."""
    sb = max(0, n // SUPER_BITS - 1)
    blk = torch.arange(SUPER_BLOCKS + 1, dtype=torch.int64, device=dev) * BLOCK_BITS + sb * SUPER_BITS
    sbs = torch.arange(n // SUPER_BITS + 2, dtype=torch.int64, device=dev) * SUPER_BITS
    pos = torch.cat([_i64([0, 1, n - 1, n, n + 7], dev), blk - 1, blk, blk + 1, sbs - 1, sbs, sbs + 1,
                     torch.randint(0, n + 1, (4096,), generator=g, device=dev)])
    return pos[(pos >= 0) & (pos <= n + 7)]


def _select_queries(ones, g, dev):
    """0, 1, ones, ones + 1, every multiple 4096 j of the select sample and its neighbours, random k."""
    j = torch.arange(1, ones // SELECT_SAMPLE + 2, dtype=torch.int64, device=dev) * SELECT_SAMPLE
    parts = [_i64([0, 1, ones, ones + 1, ones + 9], dev), j - 1, j, j + 1]
    if ones:
        parts.append(torch.randint(1, ones + 1, (4096,), generator=g, device=dev))
    k = torch.cat(parts)
    return k[k >= 0]


def _select_want(b01, k, ones):
    n = b01.numel()
    want = torch.where(k == 0, torch.zeros_like(k), torch.full_like(k, n))
    live = (k >= 1) & (k <= ones)
    if bool(live.any()):
        want[live] = R.bits_select(b01, k[live])
    return want


def _check_bitvector(E, bits, seed):
    dev = bits.device
    n = bits.numel()
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    b01 = (bits != 0).to(torch.uint8) if n and int(bits.max()) > 1 else bits
    ones = int(torch.count_nonzero(b01))
    bv = E.DeviceBitVector(bits)
    assert bv.ones == ones
    for a, b in R._chunks(n, UNPACK_CHUNK):
        _assert_same(bv.bv_bits(0, a, b - a), b01[a:b], f"bits [{a}, {b})")
    pos = _rank_positions(n, g, dev)
    _assert_same(bv.bv_rank(0, pos), R.bits_rank(b01, pos.clamp(max=n)), "rank")
    # rank_range: a window across the first superblock edge (or the middle), and one that ends at n
    mid = SUPER_BITS if n > SUPER_BITS else n // 2
    for begin in (max(0, mid - 3000), max(0, n + 1 - 5000)):
        count = min(6000, n + 1 - begin)
        want = R.bits_rank(b01, torch.arange(begin, begin + count, device=dev)).to(torch.int32)
        _assert_same(bv.bv_rank_range(0, begin, count), want, f"rank_range from {begin}")
    k = _select_queries(ones, g, dev)
    _assert_same(bv.bv_select(0, k), _select_want(b01, k, ones), "select")
    return bv


@gpu
@pytest.mark.parametrize("n,kind", BV_CASES, ids=[f"{n}-{k}" for n, k in BV_CASES])
def test_bitvector_rank_select_unpack(E, cuda, n, kind):
    # input, its 0/1 copy, the blob (n / 7 bytes) and the references' chunk temporaries
    _need_memory(cuda, 2 * n + n // 7 + 3 * GB, f"bit-vector of {n} bits")
    bits = _bv_input(kind, n, 1000 + BV_CASES.index((n, kind)), cuda)
    _check_bitvector(E, bits, seed=n % 9973)


@gpu
@pytest.mark.parametrize("n", [PACK_TILE_BITS + 1, "materialize_max+1001"])
def test_dropin_succinct_rank_select(E, cuda, n):
    """SuccinctRankSelect (csa/wavelet_tree.py) on the same kind of bits, below and above views.MATERIALIZE_MAX (a
    materialised rank_support, or one rank kernel per call): rank at block / superblock / sample edges, rank(-1),
    IndexError past n, select at the sample edges and past the ones."""
    from csa.wavelet_tree import SuccinctRankSelect
    from hkcsa import views
    if n == "materialize_max+1001":
        n = views.MATERIALIZE_MAX + 1001
    g = torch.Generator(device=cuda).manual_seed(n)
    bits = _bernoulli(n, 0.3, g, cuda).cpu().numpy()
    rs = O.rank_support(bits)
    ones = int(rs[-1])
    s = SuccinctRankSelect(bits)
    edges = {0, 1, BLOCK_BITS - 1, BLOCK_BITS, BLOCK_BITS + 1, PACK_TILE_BITS, n - 1, n}
    for i in sorted(edges | set(torch.randint(0, n + 1, (60,), generator=g, device=cuda).tolist())):
        assert int(s.rank(i)) == int(rs[i]), i
    assert int(s.rank(-1)) == ones
    with pytest.raises(IndexError):
        s.rank(n + 1)
    for k in sorted({0, 1, SELECT_SAMPLE - 1, SELECT_SAMPLE, SELECT_SAMPLE + 1, 2 * SELECT_SAMPLE, ones - 1, ones,
                     ones + 1, ones + 100}):
        assert s.select(k) == O.select(rs, k), k


# ------------------------------------------------------------------ RRR class / offset code
RRR_SCAN_BITS = RRR_SB_BITS * SCAN               # 983040 bits: exactly one iteration of rrr_scan_kernel


def _rrr_input(kind, n, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    if kind == "mixed":                          # density steps 0, 1/16 .. 1 per superblock: every class occurs
        out = torch.empty(n, dtype=torch.uint8, device=dev)
        for a, b in R._chunks(n, 1 << 26):
            p = (torch.arange(a, b, device=dev) // RRR_SB_BITS % 17).float() / 16
            out[a:b] = torch.rand(b - a, generator=g, device=dev) < p
        return out
    if kind == "random":
        return _bernoulli(n, 0.5, g, dev)
    if kind == "sparse":
        return _bernoulli(n, 1e-4, g, dev)
    if kind == "ones":
        return torch.ones(n, dtype=torch.uint8, device=dev)
    if kind == "zeros":
        return torch.zeros(n, dtype=torch.uint8, device=dev)
    raise ValueError(kind)


def _rrr_rank_positions(n, g, dev):
    """Every position from 40 before superblock 1023 to 40 past superblock 1025, block edges +-1 of the first
    superblocks, random positions, and positions past n (clamped by the kernel)."""
    window = torch.arange(RRR_SB_BITS * 1023 - 40, RRR_SB_BITS * 1026 + 40, device=dev)
    edges = torch.arange(0, 3 * RRR_SB_BITS + 1, RRR_B, device=dev)
    pos = torch.cat([window, edges - 1, edges, edges + 1, torch.randint(0, n + 1, (8192,), generator=g, device=dev),
                     _i64([0, n - 1, n, n + 1, n + RRR_B, n + 5000, 1 << 40], dev)])
    return pos[pos >= 0].unique()


def _check_rrr(vec, b01, seed, what):
    """Plan fields against rrr_expected, decode of the whole vector and of ranges at block / superblock edges, rank."""
    dev = b01.device
    n = b01.numel()
    g = torch.Generator(device=dev).manual_seed(seed)
    exp = S.rrr_expected(b01)
    got = {k: int(getattr(vec.plan, k)) for k in exp}
    assert got == exp, f"{what}: plan {got} vs {exp}"
    _assert_same(vec.bits(), b01, f"{what}: bits()")
    for begin in (0, 14, 15, 16, RRR_SB_BITS - 1, RRR_SB_BITS, RRR_SB_BITS + 1, RRR_SCAN_BITS - 961,
                  RRR_SCAN_BITS - 1, RRR_SCAN_BITS, RRR_SCAN_BITS + 1, n - 2000, n - 961, n - 16, n - 15, n - 1, n):
        if not 0 <= begin <= n:
            continue
        for count in (1, 15, 961, 2000):
            count = min(count, n - begin)
            _assert_same(vec.bits(begin, count), b01[begin:begin + count], f"{what}: bits({begin}, {count})")
    pos = _rrr_rank_positions(n, g, dev)
    _assert_same(vec.rank(pos), R.bits_rank(b01, pos.clamp(max=n)), f"{what}: rank")


RRR_CASES = ([(RRR_SCAN_BITS - 7 + r, "mixed") for r in range(RRR_B)]          # every n mod 15; nsuper 1024 / 1025
             + [(RRR_SB_BITS * 2048 + 7, k) for k in ("mixed", "random", "sparse")]
             + [(MAX_N, k) for k in ("random", "ones", "zeros", "sparse")])


@gpu
@pytest.mark.parametrize("n,kind", RRR_CASES, ids=[f"{n}-{k}" for n, k in RRR_CASES])
def test_rrr_bitvector(E, cuda, n, kind):
    # input, the decoded copy, the bit-vector blob and the code (about n / 7 bytes each), reference temporaries
    _need_memory(cuda, 2 * n + 2 * (n // 7) + 3 * GB, f"RRR vector of {n} bits")
    bits = _rrr_input(kind, n, 2000 + RRR_CASES.index((n, kind)), cuda)
    bv = E.DeviceBitVector(bits)
    vec = E.RrrVector.encode(bv, 0)
    del bv
    _check_rrr(vec, bits, n % 9973, f"{kind} n={n}")
    if kind == "ones":                # full blocks take no offset bits; only the zero-padded last block does
        assert int(vec.plan.stream_bits) == int(S.rrr_class_widths()[n % RRR_B])


@gpu
@pytest.mark.parametrize("copies", [1, 3])
def test_rrr_every_block_pattern(E, cuda, copies):
    """The 32768 15-bit patterns, each once (512 superblocks), and three copies (1536 superblocks, past one scan
    iteration): decoding reads every pattern / offset_of table entry; rank at every block edge."""
    bits = S.all_patterns_vector(cuda).repeat(copies)
    vec = E.RrrVector.encode(E.DeviceBitVector(bits), 0)
    _check_rrr(vec, bits, copies, f"all patterns x{copies}")
    edges = torch.arange(0, bits.numel() + 1, RRR_B, device=cuda)
    pos = torch.cat([edges, edges[1:] - 1, edges[:-1] + 7])
    _assert_same(vec.rank(pos), R.bits_rank(bits, pos), "rank at every block")


@gpu
def test_rrr_coded_wavelet_levels_restore_the_blob(E, cuda):
    """A wavelet tree over 2.5 * 10^6 symbols (levels of ~2600 superblocks): every level coded, checked, and restored
    through wt_from_coded_levels into rank blocks, superblocks and select samples identical to the original's; then a
    level prefix whose end falls inside a 15-bit block and inside a 224-bit rank block."""
    n = 2_500_000
    wt = E.DeviceWaveletTree(E.gen_text(E.ENG96, 17, n, cuda))
    assert wt.levels >= 2 and wt.level_len(0) > RRR_SB_BITS * 2 * SCAN
    coded = []
    for level in range(wt.levels):
        n_l = wt.level_len(level)
        vec = E.RrrVector.encode(wt, level)
        _check_rrr(vec, wt.bv_bits(level, 0, n_l), level, f"level {level}")
        coded.append(vec)
    back = E.wt_from_coded_levels(wt.plan, coded, cuda)
    lv = int(wt.plan.off_blocks[0])
    _assert_same(back.blob[lv:], wt.blob[lv:], "restored blob")
    nbits = RRR_SB_BITS * 1500 + 7                  # 7 bits into a block, 135 bits into a rank block
    assert nbits % RRR_B == 7 and nbits % BLOCK_BITS not in (0, 1) and nbits < wt.level_len(0)
    for level in range(wt.levels):
        if nbits < wt.level_len(level):
            vec = E.RrrVector.encode(wt, level, nbits)
            _check_rrr(vec, wt.bv_bits(level, 0, nbits), level, f"prefix of level {level}")


# ------------------------------------------------------------------ Golomb run code
GOLOMB_M = [1, 2, 3, 7, 31, 32, 33, 61, 62]
GOLOMB_CHUNKS = [31, 32, 33, SCAN - 1, SCAN, SCAN + 1, 2 * SCAN + 1]


def _golomb_input(kind, chunks, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    if kind == "runs":
        # a partial last chunk; runs that cross chunk 31 -> 32 (a warp edge of the carry scan), cover chunks
        # 1000 .. 1100 (warp edges and the 1024-chunk iteration edge), and end the vector
        n = chunks * GOLOMB_CHUNK - 5
        bits = _bernoulli(n, 0.2, g, dev)
        half = GOLOMB_CHUNK // 2
        for a, b in ((31 * GOLOMB_CHUNK + half, 32 * GOLOMB_CHUNK + half),
                     (1000 * GOLOMB_CHUNK - 50, 1101 * GOLOMB_CHUNK + 50),
                     ((chunks - 3) * GOLOMB_CHUNK + 17, n)):
            bits[min(a, n):min(b, n)] = 1
        return bits
    n = chunks * GOLOMB_CHUNK
    return _bernoulli(n, {"random": 0.5, "sparse": 0.003}[kind], g, dev)


def _check_golomb(bv, level, nbits, bits, m, what):
    got = bv.golomb(level, nbits, m)
    want, total = S.golomb_encode(bits, m)
    assert got.numel() == total, f"{what} m={m}: {got.numel()} code bits, want {total}"
    _assert_same(got, want, f"{what} m={m}")
    if bits.numel() <= ORACLE_MAX:
        assert np.array_equal(got.cpu().numpy(), O.golomb_encode(bits.cpu().numpy(), m)), f"{what} m={m}: oracle"


GOLOMB_CASES = [(c, k) for c in GOLOMB_CHUNKS for k in ("runs", "random", "sparse")]


@gpu
@pytest.mark.parametrize("chunks,kind", GOLOMB_CASES, ids=[f"{c}chunks-{k}" for c, k in GOLOMB_CASES])
def test_golomb_chunk_carries(E, cuda, chunks, kind):
    bits = _golomb_input(kind, chunks, 3000 + GOLOMB_CASES.index((chunks, kind)), cuda)
    bv = E.DeviceBitVector(bits)
    for m in GOLOMB_M:
        _check_golomb(bv, 0, bits.numel(), bits, m, f"{kind} {chunks} chunks")


GOLOMB_MAX_CASES = [("ones", 1), ("ones", 30), ("ones", 62), ("random", 2), ("sparse", 30)]


@gpu
@pytest.mark.parametrize("kind,m", GOLOMB_MAX_CASES, ids=[f"{k}-m{m}" for k, m in GOLOMB_MAX_CASES])
def test_golomb_at_the_size_limit(E, cuda, kind, m):
    """2^30 - 2 bits: all ones is one run closed by the end of input (its code is v // m zeros, a one and m bits);
    random bits hold ~2^28 runs, whose per-run arrays dominate the reference's memory."""
    n = MAX_N
    runs = {"ones": 1, "random": n // 4 + 1, "sparse": n // 10 ** 5 + 1}[kind]
    code = {"ones": n // m + 1 + m, "random": n, "sparse": runs * (m + 1)}[kind]
    # input, blob, device code and reference code, per-run int64 arrays (starts, ends, lengths, offsets, ...)
    _need_memory(cuda, n + n // 7 + 2 * code + 64 * runs + 3 * GB, f"Golomb code of {n} {kind} bits")
    g = torch.Generator(device=cuda).manual_seed(4000 + m)
    bits = {"ones": lambda: torch.ones(n, dtype=torch.uint8, device=cuda),
            "random": lambda: _bernoulli(n, 0.5, g, cuda),
            "sparse": lambda: _bernoulli(n, 1e-5, g, cuda)}[kind]()
    bv = E.DeviceBitVector(bits)
    _check_golomb(bv, 0, n, bits, m, f"{kind} 2^30-2")


@gpu
def test_golomb_level_prefixes_ending_inside_a_run(E, cuda):
    """WaveletTree.build_tree asks for the code of a level prefix (the left-most node).  Prefixes that end inside runs
    of ones of level 0, in the first and the second 1024-chunk iteration, on a sequence of long symbol runs."""
    g = torch.Generator(device=cuda).manual_seed(77)
    runs = 3000
    sym = torch.tensor(list(b"abcd"), dtype=torch.uint8, device=cuda)[torch.randint(0, 4, (runs,), generator=g,
                                                                                    device=cuda)]
    lens = torch.randint(1, 4000, (runs,), generator=g, device=cuda)
    seq = torch.repeat_interleave(sym, lens)
    seq[:4] = sym.new_tensor(list(b"abcd"))
    wt = E.DeviceWaveletTree(seq)
    n0 = wt.level_len(0)
    assert n0 > 2 * SCAN * GOLOMB_CHUNK
    level0 = wt.bv_bits(0, 0, n0)
    starts, lengths = S.ones_runs(level0)
    pick = ((lengths >= 3) & (starts + lengths < n0)).nonzero().flatten()
    pick = pick[torch.linspace(0, pick.numel() - 1, 12, device=cuda).long()]
    for r in pick.tolist():
        nbits = int(starts[r] + lengths[r] // 2)
        for m in (1, 3, 30, 62):
            _check_golomb(wt, 0, nbits, level0[:nbits], m, f"level-0 prefix of {nbits} bits")


# ------------------------------------------------------------------ refusals
def _plan(levels, level_len):
    p = _lib.WtPlan()
    p.levels = levels
    p.level_len[0] = level_len
    return p


def test_refusals_before_any_device_access():
    """Argument checks that come before any device access: no kernel is launched and the outputs are untouched."""
    L = _lib.load()
    before = L.hkcsa_launch_count()
    p = _lib.WtPlan()
    assert L.hkcsa_bitvec_plan(MAX_N + 1, C.byref(p)) == _lib.ERANGE
    assert L.hkcsa_bitvec_plan(MAX_N, C.byref(p)) == _lib.OK and p.level_len[0] == MAX_N
    # a host-made plan of one level of 2^30 bits: the coded form's 32-bit superblock entries take at most MAX_N + 1
    wt = _plan(1, MAX_N + 2)
    rp = _lib.RrrPlan()
    assert L.hkcsa_rrr_encode(1, C.byref(wt), 0, MAX_N + 2, 1, C.byref(rp), None, 0, 1, 1 << 20, None) == _lib.ERANGE
    gp = _plan(1, 1000)
    out_bits = C.c_uint64(12345)
    for level, nbits, m in ((0, 1000, 0), (0, 1000, 63), (0, 1001, 7), (1, 10, 7)):
        rc = L.hkcsa_golomb_encode(1, C.byref(gp), level, nbits, m, None, 0, C.byref(out_bits), 1, 1 << 20, None)
        assert rc == _lib.EINVAL, (level, nbits, m)
        assert out_bits.value == 12345
    assert L.hkcsa_launch_count() == before


@gpu
def test_refusals_on_the_device(E, cuda):
    """A Golomb output one byte short: ESCRATCH after the sizing pass (which has to run to know the size), no kernel
    beyond it, nothing written.  An RRR output 8 bytes off 32-byte alignment: EINVAL before any launch."""
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    n = 5 * GOLOMB_CHUNK + 3
    bits = (torch.arange(n, device=cuda) % 5 != 0).to(torch.uint8)
    bv = E.DeviceBitVector(bits)
    nscr = L.hkcsa_golomb_scratch_bytes(n)
    scratch = torch.empty(nscr, dtype=torch.uint8, device=cuda)
    total = C.c_uint64(0)
    before = L.hkcsa_launch_count()
    _lib.check(L.hkcsa_golomb_encode(bv.blob.data_ptr(), C.byref(bv.plan), 0, n, 3, None, 0, C.byref(total),
                                     scratch.data_ptr(), nscr, st))
    sizing = L.hkcsa_launch_count() - before
    want, size = S.golomb_encode(bits, 3)
    assert total.value == size
    out = torch.full((size,), 0xAB, dtype=torch.uint8, device=cuda)
    before = L.hkcsa_launch_count()
    rc = L.hkcsa_golomb_encode(bv.blob.data_ptr(), C.byref(bv.plan), 0, n, 3, out.data_ptr(), size - 1,
                               C.byref(total), scratch.data_ptr(), nscr, st)
    assert rc == _lib.ESCRATCH
    assert L.hkcsa_launch_count() - before == sizing
    torch.cuda.synchronize()
    assert bool((out == 0xAB).all())
    _lib.check(L.hkcsa_golomb_encode(bv.blob.data_ptr(), C.byref(bv.plan), 0, n, 3, out.data_ptr(), size,
                                     C.byref(total), scratch.data_ptr(), nscr, st))
    _assert_same(out, want, "golomb with the exact capacity")

    tab = E.rrr_tables(cuda)
    nscr = L.hkcsa_rrr_scratch_bytes(n)
    scratch = torch.empty(nscr, dtype=torch.uint8, device=cuda)
    blob = torch.zeros(1 << 16, dtype=torch.uint8, device=cuda)
    rp = _lib.RrrPlan()
    before = L.hkcsa_launch_count()
    rc = L.hkcsa_rrr_encode(bv.blob.data_ptr(), C.byref(bv.plan), 0, n, tab.data_ptr(), C.byref(rp),
                            blob.data_ptr() + 8, blob.numel() - 8, scratch.data_ptr(), nscr, st)
    assert rc == _lib.EINVAL and b"aligned" in L.hkcsa_last_error()
    assert L.hkcsa_launch_count() == before
    torch.cuda.synchronize()
    assert not bool(blob.any())
