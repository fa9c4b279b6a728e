"""The two sort primitives of csrc/radix_sort.cu, called through the C-ABI and checked pair by pair against an exact
stable sort computed by torch on the device:

* hkcsa_sort_pairs_u64, the onesweep LSD sort of (u64 key, u32 value) pairs behind round 0 and every refinement round
  of both suffix-array builders: both tile shapes and every ragged-tail class of the last tile, 1 to 8 passes (odd
  counts end with the copy back from the alternate buffers), random bits above `key_bits` that are sorted up to the
  next digit and carried unchanged beyond it, key distributions aimed at the histogram fast path, the padding key and
  the look-back, a scratch region that starts out dirty and is reused, and n = 2^30 - 2, where the 30-bit look-back
  counts come within one of their limit.
* radix_partition_bytes, the byte onesweep on 8192-byte tiles, through hkcsa_partition_bytes (the drop-in
  WaveletTree's next_text) and hkcsa_symbol_positions (FMIndex.precompute_rank): tile edges, LUTs that send real
  bytes to bucket 255 (the digit of the last tile's padding slots), sizes up to 2^30 - 2.

Every output buffer starts out holding something other than the answer, so a slot the kernel never writes fails the
comparison.  The argument checks that need no device run without the gpu mark."""
import ctypes as C

import numpy as np
import pytest
import torch

from hkcsa import _lib

gpu = pytest.mark.gpu

# Tile shapes of the sorts under test -- keep in step with radix_sort.cu:554-555 (run_onesweep64<448, 2, 16> from
# 2^22 pairs on, run_onesweep64<384, 3> with OS_IPT = 8 below) and radix_sort.cuh:26-28 (SORT8_THREADS x SORT8_IPT).
SORT_SMALL_TILE = 384 * 8            # pairs per tile below the switch
SORT_LARGE_TILE = 448 * 16           # pairs per tile from the switch on
SORT_LARGE_MIN_N = 1 << 22           # the switch
BYTE_TILE = 256 * 32                 # bytes per tile of the byte partition

MAX_N = _lib.MAX_N                   # 2^30 - 2
LB_VAL = (1 << 30) - 1               # look-back counts are 30 bits (radix_sort.cuh)
INT64_MIN = -(1 << 63)
KEY_SENTINEL = 0x5A5A_5A5A_5A5A_5A5A  # alternate-buffer fill: no generated key below equals it
GB = 1 << 30


def _tile_of(n):
    return SORT_LARGE_TILE if n >= SORT_LARGE_MIN_N else SORT_SMALL_TILE


def _i64(u):
    """An unsigned 64-bit pattern as the int64 torch stores."""
    u &= (1 << 64) - 1
    return u - (1 << 64) if u >> 63 else u


def _passes(key_bits):
    return (key_bits + 7) // 8


def _need_memory(dev, need, what):
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need:
        pytest.skip(f"{what}: needs {need / GB:.1f} GiB of device memory, {free / GB:.1f} GiB free")


def _assert_same(got, want, what):
    assert got.dtype == want.dtype and got.shape == want.shape, f"{what}: {got.dtype}{tuple(got.shape)} vs " \
                                                               f"{want.dtype}{tuple(want.shape)}"
    if torch.equal(got, want):
        return
    bad = (got != want).nonzero().flatten()
    i = int(bad[0])
    lo, hi = max(0, i - 2), min(got.numel(), i + 3)
    raise AssertionError(f"{what}: {bad.numel()} of {got.numel()} slots differ, first at {i}: "
                         f"got {got[lo:hi].tolist()}, want {want[lo:hi].tolist()} (slots {lo}..{hi - 1})")


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


# ------------------------------------------------------------------ (u64, u32) pairs: inputs and reference
def _rand64(n, g, dev):
    return torch.empty(n, dtype=torch.int64, device=dev).random_(INT64_MIN, None, generator=g)


def _carried_garbage(n, key_bits, g, dev):
    """Random bits from bit 8 * passes up (zero below): bits the sort carries but never looks at."""
    p = _passes(key_bits)
    if p == 8:
        return torch.zeros(n, dtype=torch.int64, device=dev)
    return _rand64(n, g, dev) & _i64(~((1 << (8 * p)) - 1))


def _spread(n, key_bits, dev):
    """0 .. 2^key_bits - 1, non-decreasing over n slots, as int64 bit patterns."""
    i = torch.arange(n, dtype=torch.int64, device=dev)
    width = max(1, (n - 1).bit_length())
    if key_bits >= width:
        return i << (key_bits - width)
    return (i << key_bits) // n


def _keys(dist, n, key_bits, g, dev):
    """n 64-bit keys for a sort on `key_bits` bits.  Bits above key_bits are never zero across the array: `random`
    draws all 64 bits (so the bits between key_bits and the next digit boundary are sorted on too), the structured
    distributions either draw whole 64-bit keys per group of equal keys or add random bits above the sorted digits."""
    p = _passes(key_bits)
    garbage = lambda: _carried_garbage(n, key_bits, g, dev)                       # noqa: E731
    if dist == "random":
        return _rand64(n, g, dev)
    if dist == "equal":                        # one key: one digit per tile and pass, warp-uniform histogram path
        return _rand64(1, g, dev).expand(n).clone()
    if dist == "all_ones":                     # every real key equals the last tile's padding key
        return torch.full((n,), -1, dtype=torch.int64, device=dev)
    if dist == "two":                          # two keys that differ in the lowest and the highest sorted bit
        a = _rand64(1, g, dev)
        b = a ^ _i64(1 | (1 << (key_bits - 1)))
        pick = torch.randint(0, 2, (n,), generator=g, device=dev, dtype=torch.int64).bool()
        return torch.where(pick, a, b) ^ garbage()
    if dist.startswith("runs"):                # runs of equal whole keys: warp-aligned (32) and misaligned (31, 33)
        run = int(dist[4:])
        ids = torch.arange(n, dtype=torch.int64, device=dev) // run
        return _rand64((n + run - 1) // run, g, dev)[ids]
    if dist == "ascending":
        return _spread(n, key_bits, dev) ^ garbage()
    if dist == "descending":
        return (_i64((1 << key_bits) - 1) - _spread(n, key_bits, dev)) ^ garbage()
    if dist == "tile_edges":                   # one whole key per tile: every digit changes exactly at tile edges
        tile = _tile_of(n)
        ids = torch.arange(n, dtype=torch.int64, device=dev) // tile
        return _rand64((n + tile - 1) // tile, g, dev)[ids]
    if dist in ("top_only", "bottom_only"):   # only the last (first) pass sees more than one digit
        sh = 8 * (p - 1) if dist == "top_only" else 0
        c = _rand64(1, g, dev) & _i64(~(0xFF << sh))
        d = torch.randint(0, 256, (n,), generator=g, device=dev, dtype=torch.int64)
        return (c | (d << sh)) ^ garbage()
    raise ValueError(dist)


def _vals(kind, n, g, dev):
    if kind == "identity":                     # stability shows directly
        return torch.arange(n, dtype=torch.int32, device=dev)
    return torch.randperm(n, generator=g, device=dev).to(torch.int32)   # each value must travel with its own key


def _expected(keys, vals, key_bits):
    """Stable sort on key mod 2^(8 * passes), unsigned; the full 64-bit keys and the values follow."""
    p = _passes(key_bits)
    sk = keys.clone() if p == 8 else keys & ((1 << (8 * p)) - 1)
    sk ^= INT64_MIN                            # unsigned order as signed order
    idx = torch.sort(sk, stable=True).indices
    del sk
    return keys[idx], vals[idx]


def _scratch(n, dev):
    """Scratch for hkcsa_sort_pairs_u64, filled with 0xFF: the sort must clear what it relies on."""
    return torch.full((_lib.load().hkcsa_sort_scratch_bytes(n),), 0xFF, dtype=torch.uint8, device=dev)


def _sort(keys, vals, key_bits, scratch=None):
    """hkcsa_sort_pairs_u64 in place on (keys, vals), with alternate buffers filled with sentinels and a dirty
    scratch; returns the alternate buffers."""
    L = _lib.load()
    n = keys.numel()
    k_alt = torch.full_like(keys, KEY_SENTINEL)
    v_alt = torch.full_like(vals, -1)
    if scratch is None:
        scratch = _scratch(n, keys.device)
    _lib.check(L.hkcsa_sort_pairs_u64(keys.data_ptr(), vals.data_ptr(), k_alt.data_ptr(), v_alt.data_ptr(), n,
                                      key_bits, scratch.data_ptr(), scratch.numel(),
                                      torch.cuda.current_stream().cuda_stream))
    return k_alt, v_alt


def _check_sort(dev, n, key_bits, dist, values, seed, scratch=None):
    g = torch.Generator(device=dev).manual_seed(seed)
    keys = _keys(dist, n, key_bits, g, dev)
    vals = _vals(values, n, g, dev)
    assert not bool((keys == KEY_SENTINEL).any())
    want_k, want_v = _expected(keys, vals, key_bits)
    k_alt, v_alt = _sort(keys, vals, key_bits, scratch)
    what = f"n={n} key_bits={key_bits} {dist} {values}"
    _assert_same(keys, want_k, f"{what}: keys")
    _assert_same(vals, want_v, f"{what}: values")
    # The alternate buffers hold the output of the last odd-numbered pass (and, for odd pass counts, the result the
    # sort copied back): no sentinel may survive in them.
    assert not bool((v_alt == -1).any()), f"{what}: a slot of the alternate values was never written"
    if _passes(key_bits) % 2:
        _assert_same(k_alt, want_k, f"{what}: alternate keys")
        _assert_same(v_alt, want_v, f"{what}: alternate values")


# ------------------------------------------------------------------ tile shapes and ragged tails
def _tail_sizes():
    out = []
    for tile, qs in ((SORT_SMALL_TILE, (1, 20)), (SORT_LARGE_TILE, (586, 601))):
        for q in qs:
            for r in (0, 1, 2, 3, 4, 5, tile - 1):
                n = q * tile + r
                assert _tile_of(n) == tile, (tile, q, r)
                out.append(n)
    return out


@gpu
@pytest.mark.parametrize("key_bits,values", [(16, "identity"), (40, "permutation")])
@pytest.mark.parametrize("n", _tail_sizes())
def test_sort_pairs_tile_tails(E, cuda, n, key_bits, values):
    """n = q * TILE + r: the last tile holds r pairs (TILE for r = 0), so nvalid mod 4 takes every class and the TMA
    load finishes 0 or 1 key and 0 to 3 values one by one; two and five passes."""
    _check_sort(cuda, n, key_bits, "random", values, seed=n % 100_003 + key_bits)


@gpu
@pytest.mark.parametrize("n,key_bits,values", [
    (SORT_LARGE_MIN_N - 1, 64, "permutation"), (SORT_LARGE_MIN_N - 1, 20, "identity"),
    (SORT_LARGE_MIN_N, 64, "permutation"), (SORT_LARGE_MIN_N, 20, "identity"),
    (10 ** 8, 40, "permutation"), (10 ** 8, 64, "identity")])
def test_sort_pairs_switch_and_large(E, cuda, n, key_bits, values):
    """Both sides of the tile-shape switch, and 10^8 pairs (the C2 workload's size)."""
    _check_sort(cuda, n, key_bits, "random", values, seed=7 + key_bits)


# ------------------------------------------------------------------ key widths and distributions
KEY_BITS = (1, 7, 8, 9, 16, 20, 24, 40, 48, 56, 63, 64)
DISTS = ("random", "equal", "all_ones", "two", "runs31", "runs32", "runs33", "ascending", "descending", "tile_edges",
         "top_only", "bottom_only")
WIDTH_SIZES = {"small_tile": (37 * SORT_SMALL_TILE + 3, "identity"),
               "large_tile": (590 * SORT_LARGE_TILE + 2, "permutation")}


@gpu
@pytest.mark.parametrize("shape", sorted(WIDTH_SIZES))
@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("key_bits", KEY_BITS)
def test_sort_pairs_key_widths(E, cuda, key_bits, dist, shape):
    """1 to 8 passes, odd and even, with bits above key_bits set: the order is that of key mod 2^(8 * passes) and
    every key comes back with all 64 bits."""
    n, values = WIDTH_SIZES[shape]
    _check_sort(cuda, n, key_bits, dist, values, seed=1000 * key_bits + DISTS.index(dist))


def test_distributions_hit_their_targets():
    """The generators make what the distribution names promise (checked on the host, small n)."""
    dev = torch.device("cpu")
    n, kb = 3 * SORT_SMALL_TILE + 5, 20
    for dist in DISTS:
        g = torch.Generator(device=dev).manual_seed(1)
        keys = _keys(dist, n, kb, g, dev)
        assert keys.shape == (n,) and keys.dtype == torch.int64
        assert bool((keys & _i64(~((1 << kb) - 1)) != 0).any()), f"{dist}: no bits above key_bits"
    g = torch.Generator(device=dev).manual_seed(1)
    assert torch.unique(_keys("equal", n, kb, g, dev)).numel() == 1
    assert bool((_keys("all_ones", n, kb, g, dev) == -1).all())
    low = _keys("two", n, kb, g, dev) & ((1 << 24) - 1)
    assert torch.unique(low).numel() == 2
    for run in (31, 32, 33):
        k = _keys(f"runs{run}", n, kb, g, dev)
        assert bool((k[:run] == k[0]).all()) and int(k[run]) != int(k[0])
    asc = _keys("ascending", n, kb, g, dev) & ((1 << kb) - 1)
    assert bool((asc[1:] >= asc[:-1]).all()) and int(asc[-1]) > int(asc[0])
    desc = _keys("descending", n, kb, g, dev) & ((1 << kb) - 1)
    assert bool((desc[1:] <= desc[:-1]).all())
    k = _keys("tile_edges", n, kb, g, dev)
    assert bool((k[:SORT_SMALL_TILE] == k[0]).all()) and int(k[SORT_SMALL_TILE]) != int(k[0])
    for dist, sh in (("top_only", 16), ("bottom_only", 0)):
        k = _keys(dist, n, kb, g, dev) & ((1 << 24) - 1)
        assert torch.unique(k & ~(0xFF << sh)).numel() == 1 and torch.unique(k >> sh & 0xFF).numel() > 1
    # the reference orders unsigned: all-ones sorts last, and only the sorted digits count
    keys = torch.tensor([-1, 0, _i64(1 << 63), 1 << 40, 1], dtype=torch.int64)
    vals = torch.arange(5, dtype=torch.int32)
    assert _expected(keys, vals, 64)[1].tolist() == [1, 4, 3, 2, 0]
    assert _expected(keys, vals, 40)[1].tolist() == [1, 2, 3, 4, 0]   # 5 passes: bit 40 is carried, not sorted
    assert _expected(keys, vals, 41)[1].tolist() == [1, 2, 4, 3, 0]   # 6 passes: bit 40 is sorted on


# ------------------------------------------------------------------ scratch reuse
@gpu
@pytest.mark.parametrize("order", ["large_then_small", "small_then_large"])
def test_sort_pairs_reuses_one_dirty_scratch(E, cuda, order):
    """One scratch region, filled with 0xFF once, serves sorts of different n and width in turn, as in the builders'
    rounds (look-back halves and tickets of the previous sort left behind)."""
    runs = [(590 * SORT_LARGE_TILE + 5, 64, "random", "permutation"),
            (3 * SORT_SMALL_TILE + 2, 20, "runs33", "identity"),
            (2 * SORT_SMALL_TILE + 1, 40, "tile_edges", "permutation")]
    if order == "small_then_large":
        runs = runs[::-1]
    scratch = _scratch(max(r[0] for r in runs), cuda)
    for k, (n, key_bits, dist, values) in enumerate(runs):
        _check_sort(cuda, n, key_bits, dist, values, seed=50 + k, scratch=scratch)


# ------------------------------------------------------------------ the size limit
def _sort_limit_need(n):
    """keys + values (12 B/pair) beside the reference's peak: its masked keys, the index iota, the sorted keys and
    indices and the sort's double buffers (48 B).  The expected copies and the alternate buffers (24 B) come later,
    when the reference's temporaries are gone.  Plus the sort scratch (look-back table)."""
    return 60 * n + _lib.load().hkcsa_sort_scratch_bytes(n) + 2 * GB


@gpu
@pytest.mark.parametrize("dist,values", [("equal", "permutation"), ("random", "permutation")])
def test_sort_pairs_at_the_size_limit(E, cuda, dist, values):
    """n = 2^30 - 2 with 40-bit keys (the DNA round-0 width, five passes) and random bits above bit 40.  With all keys
    equal one digit takes every pair in every pass: the look-back prefixes grow by a whole tile per tile, and the last
    tile's inclusive count is n, one below the largest count a 30-bit look-back entry holds."""
    n = MAX_N
    assert n < LB_VAL
    _need_memory(cuda, _sort_limit_need(n), f"sort of {n} pairs")
    _check_sort(cuda, n, 40, dist, values, seed=30 + len(dist))
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ refusals
def _sort_rc(n, key_bits, keys=None, vals=None, k_alt=None, v_alt=None, scratch=None, scratch_bytes=0):
    L = _lib.load()
    p = lambda t: None if t is None else t.data_ptr()      # noqa: E731
    return L.hkcsa_sort_pairs_u64(p(keys), p(vals), p(k_alt), p(v_alt), n, key_bits, p(scratch), scratch_bytes, None)


def test_sort_pairs_refuses_bad_sizes_and_widths():
    """Checked before any pointer is looked at, so they run without a device; nothing is launched."""
    L = _lib.load()
    before = L.hkcsa_launch_count()
    assert _sort_rc(MAX_N + 1, 64) == _lib.ERANGE
    assert b"HKCSA_MAX_N" in L.hkcsa_last_error()
    assert _sort_rc(1 << 32, 8) == _lib.ERANGE
    for bad in (65, 128, -1):
        assert _sort_rc(1000, bad) == _lib.EINVAL
        assert b"key_bits" in L.hkcsa_last_error()
        assert _sort_rc(0, bad) == _lib.EINVAL            # the width is checked even when there is nothing to sort
    assert _sort_rc(0, 64) == _lib.OK                     # nothing to sort: no pointer needed
    assert _sort_rc(1000, 0) == _lib.OK                   # no digit to sort on
    assert _sort_rc(MAX_N, 0) == _lib.OK
    assert L.hkcsa_launch_count() == before


@gpu
def test_sort_pairs_refuses_misaligned_buffers(E, cuda):
    """The TMA bulk copies need 16-byte aligned buffers: a buffer 8 bytes off is refused with EINVAL before anything
    is launched or written; a scratch region one byte short is refused with ESCRATCH."""
    L = _lib.load()
    n = 2 * SORT_SMALL_TILE + 3
    keys = torch.arange(n + 2, dtype=torch.int64, device=cuda)
    vals = torch.arange(n + 4, dtype=torch.int32, device=cuda)
    k_alt = torch.full((n + 2,), KEY_SENTINEL, dtype=torch.int64, device=cuda)
    v_alt = torch.full((n + 4,), -1, dtype=torch.int32, device=cuda)
    scratch = _scratch(n, cuda)
    good = dict(keys=keys[:n], vals=vals[:n], k_alt=k_alt[:n], v_alt=v_alt[:n])
    shifted = dict(keys=keys[1:n + 1], vals=vals[2:n + 2], k_alt=k_alt[1:n + 1], v_alt=v_alt[2:n + 2])
    for name in good:
        assert shifted[name].data_ptr() % 16 == 8
    torch.cuda.synchronize()
    before = L.hkcsa_launch_count()
    for name in good:
        bufs = dict(good, **{name: shifted[name]})
        assert _sort_rc(n, 64, scratch=scratch, scratch_bytes=scratch.numel(), **bufs) == _lib.EINVAL, name
        assert b"16-byte aligned" in L.hkcsa_last_error()
    assert _sort_rc(n, 64, scratch=scratch, scratch_bytes=scratch.numel() - 1, **good) == _lib.ESCRATCH
    assert L.hkcsa_launch_count() == before
    torch.cuda.synchronize()
    assert torch.equal(keys, torch.arange(n + 2, dtype=torch.int64, device=cuda))
    assert torch.equal(vals, torch.arange(n + 4, dtype=torch.int32, device=cuda))
    assert bool((k_alt == KEY_SENTINEL).all()) and bool((v_alt == -1).all())


# ------------------------------------------------------------------ byte partition
PART_SIZES = (1, 31, BYTE_TILE - 1, BYTE_TILE, BYTE_TILE + 1, 3 * BYTE_TILE + 1, 10 ** 6 + 3, 10 ** 8, MAX_N)
LUTS = ("identity", "zero", "all_255", "wavelet_filter", "random17")
INPUTS = ("uniform", "all_a", "runs")


def _bytes(kind, n, g, dev):
    if kind == "uniform":
        return torch.randint(0, 256, (n,), generator=g, device=dev, dtype=torch.uint8)
    if kind == "all_a":
        return torch.full((n,), ord("a"), dtype=torch.uint8, device=dev)
    # runs of 3001 equal bytes: 3001 and 8192 are coprime, so runs straddle tile edges at every offset
    ids = torch.arange(n, dtype=torch.int64, device=dev) // 3001
    return torch.randint(0, 256, ((n + 3000) // 3001,), generator=g, device=dev, dtype=torch.uint8)[ids]


def _lut(kind, x, seed):
    if kind == "identity":                     # 256 buckets: a counting sort of the bytes
        return np.arange(256, dtype=np.uint8)
    if kind == "zero":
        return np.zeros(256, dtype=np.uint8)
    if kind == "all_255":                      # every real byte shares the padding slots' digit
        return np.full(256, 255, dtype=np.uint8)
    if kind == "wavelet_filter":               # WaveletTree._filter: the left half of the alphabet -> 0, rest -> 255
        alpha = torch.unique(x).cpu().numpy()
        lut = np.full(256, 255, dtype=np.uint8)
        lut[alpha[:(len(alpha) + 1) // 2]] = 0
        return lut
    rng = np.random.RandomState(seed)          # 17 buckets 15 apart: empty buckets between them and after
    return rng.choice(np.arange(0, 255, 15, dtype=np.uint8), size=256)


def _partition_need(n):
    """input, output, the int32 index for the LUT lookup, the bucket of every byte, the reference's sort (keys and
    int64 indices, each twice) and the gathered expectation, plus scratch."""
    return n * (1 + 1 + 4 + 1 + 2 * (1 + 8) + 1) + 2 * _lib.load().hkcsa_partition_scratch_bytes(n) + 2 * GB


@gpu
@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("lut_kind", LUTS)
@pytest.mark.parametrize("n", PART_SIZES)
def test_partition_bytes(E, cuda, n, lut_kind, inp):
    """hkcsa_partition_bytes equals x gathered by the stable argsort of lut[x]; bucket sizes equal bincount(lut[x])."""
    if n > 10 ** 8:
        _need_memory(cuda, _partition_need(n), f"partition of {n} bytes")
    L = _lib.load()
    g = torch.Generator(device=cuda).manual_seed(n % 9973 + 17 * LUTS.index(lut_kind) + INPUTS.index(inp))
    x = _bytes(inp, n, g, cuda)
    lut = _lut(lut_kind, x, seed=n % 1000)
    bucket = torch.index_select(torch.from_numpy(lut).to(cuda), 0, x.to(torch.int32))
    want = x[torch.sort(bucket, stable=True).indices]
    want_sizes = torch.bincount(bucket, minlength=256).cpu().numpy().astype(np.uint64)
    del bucket
    out = want ^ 0xFF                          # every slot starts out wrong
    sizes = np.full(256, 7, dtype=np.uint64)
    nbytes = L.hkcsa_partition_scratch_bytes(n)
    scratch = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=cuda)
    _lib.check(L.hkcsa_partition_bytes(x.data_ptr(), n, lut.ctypes.data_as(C.POINTER(C.c_uint8)), out.data_ptr(),
                                       sizes.ctypes.data_as(C.POINTER(C.c_uint64)), scratch.data_ptr(), nbytes,
                                       torch.cuda.current_stream().cuda_stream))
    assert np.array_equal(sizes, want_sizes), f"bucket sizes differ at {np.nonzero(sizes != want_sizes)[0][:8]}"
    _assert_same(out, want, f"partition n={n} lut={lut_kind} input={inp}")
    del x, out, want, scratch
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("n", PART_SIZES)
def test_symbol_positions_exact(E, cuda, n, inp):
    """hkcsa_symbol_positions: the positions are the stable argsort of the bytes, start[] the exclusive cumulative
    sum of their histogram (257 entries)."""
    if n > 10 ** 8:
        _need_memory(cuda, _partition_need(n) + 4 * n, f"symbol positions of {n} bytes")
    L = _lib.load()
    g = torch.Generator(device=cuda).manual_seed(n % 7919 + INPUTS.index(inp))
    x = _bytes(inp, n, g, cuda)
    want = torch.sort(x, stable=True).indices.to(torch.int32)
    hist = torch.bincount(x, minlength=256)
    want_start = torch.zeros(257, dtype=torch.int64, device=cuda)
    want_start[1:] = torch.cumsum(hist, 0)
    pos = torch.full((n,), -1, dtype=torch.int32, device=cuda)
    start = torch.full((257,), -1, dtype=torch.int64, device=cuda)
    nbytes = L.hkcsa_symbol_positions_scratch_bytes(n)
    scratch = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=cuda)
    _lib.check(L.hkcsa_symbol_positions(x.data_ptr(), n, pos.data_ptr(), start.data_ptr(), scratch.data_ptr(), nbytes,
                                        torch.cuda.current_stream().cuda_stream))
    _assert_same(start, want_start, f"symbol start n={n} input={inp}")
    _assert_same(pos, want, f"symbol positions n={n} input={inp}")
    del x, pos, want, scratch
    torch.cuda.empty_cache()
