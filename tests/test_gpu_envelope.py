"""The whole single-GPU index up to its size limit, n = 2^30 - 2 (DESIGN section 2), checked against the exact torch
references of tests/device_reference.py on the device: suffix array (Burkhardt-Kaerkkaeinen checker), BWT, C[],
wavelet-tree access / rank / select across superblock boundaries, the sampled SA and LF-walk locate, count, extract,
H_k, and the compressed save / load round trip.

Sizes are those a user may hand one GPU: at 2^30 - 2 the radix-sort look-back counters (30 bits) are one below their
limit on a text whose keys all share a digit (all_a_max), and every rank directory holds ~73 superblocks, so the
absolute u64 superblock counts take part in every rank.  Repetitive texts take the eager rank scatter and up to
log2 n doubling rounds; sigma = 18 / 19 sit either side of the k-gram round-0 switch; 255 byte values take 8 levels,
64-bit keys and the phased BWT gather.

One index per text, freed before the next.  A case skips only when the device reports less free memory than its
computed peak (the number is in the reason).  HKCSA_ENVELOPE_SCALE = 2^j (default 1) divides every n, for a quick
rehearsal; the default is the sizes above."""
import os

import pytest
import torch

import device_reference as R

pytestmark = pytest.mark.gpu

SCALE = int(os.environ.get("HKCSA_ENVELOPE_SCALE", "1"))
assert SCALE >= 1 and SCALE & (SCALE - 1) == 0, "HKCSA_ENVELOPE_SCALE must be a power of two"
DOLLAR = 0x24
SUPER_BITS = 65536 * 224           # bits per rank superblock (DESIGN section 2)
BLOCK_BITS = 224
MAX_N = (1 << 30) - 2
GB = 1 << 30


def _gen(E, kind, seed, n):
    return E.gen_text(kind, seed, n)


def _uniform(m, letters, seed, dev):
    """m symbols uniform over `letters` (bytes), on the device, every letter present."""
    g = torch.Generator(device=dev).manual_seed(seed)
    alpha = torch.tensor(list(letters), dtype=torch.uint8, device=dev)
    out = alpha[torch.randint(0, len(letters), (m,), generator=g, device=dev)]
    out[: len(letters)] = alpha
    return out


def _dollar(dev):
    return torch.tensor([DOLLAR], dtype=torch.uint8, device=dev)


def _mississippi(m, dev):
    unit = torch.tensor(list(b"mississippi"), dtype=torch.uint8, device=dev)
    return unit.repeat(-(-m // 11))[:m]


# name -> (n, make(E, n, dev) -> uint8 text ending in '$', sample rate, occ layouts, sentinel unique)
def _cases():
    top = (1 << 30) // SCALE - 2
    k = ((1 << 28) // SCALE) // 12
    blk = (1 << 20) // SCALE
    no_dollar = bytes(b for b in range(256) if b != DOLLAR)
    return {
        "eng_max": (top, lambda E, n, d: torch.cat([_gen(E, E.ENG96, 42, n - 1), _dollar(d)]), 32, (1, 0), True),
        "dna_max": (top, lambda E, n, d: torch.cat([_gen(E, E.DNA4, 43, n - 1), _dollar(d)]), 32, (1,), True),
        "all_a_max": (top, lambda E, n, d: torch.cat([torch.full((n - 1,), ord("a"), dtype=torch.uint8, device=d),
                                                      _dollar(d)]), 32, (), True),
        "bytes255": ((1 << 29) // SCALE + 1, lambda E, n, d: torch.cat([_uniform(n - 1, no_dollar, 7, d), _dollar(d)]),
                     32, (), True),
        "sigma18": ((1 << 27) // SCALE, lambda E, n, d: torch.cat([_uniform(n - 1, b"abcdefghijklmnopq", 8, d),
                                                                    _dollar(d)]), 32, (1,), True),
        "sigma19": ((1 << 27) // SCALE, lambda E, n, d: torch.cat([_uniform(n - 1, b"abcdefghijklmnopqr", 9, d),
                                                                    _dollar(d)]), 32, (1,), True),
        "mississippi_inner": (12 * k + 1, lambda E, n, d: torch.cat([
            torch.tensor(list(b"mississippi$"), dtype=torch.uint8, device=d).repeat(k), _dollar(d)]), 32, (), False),
        "period11": ((1 << 28) // SCALE, lambda E, n, d: torch.cat([_mississippi(n - 1, d), _dollar(d)]), 32, (1,),
                     True),
        "block_repeat": (256 * blk + 1, lambda E, n, d: torch.cat([_gen(E, E.ENG96, 44, blk).repeat(256), _dollar(d)]),
                         32, (), True),
    }


CASES = _cases()


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _peak_bytes(n, sigma, layouts):
    """text + SA + BWT + index (~1.5 B/symbol) + the build's transient (40.5 B/symbol, DESIGN section 2), or, after the
    build, the checks: the int32 ISA and LF^-1 of the references (8 B/symbol), the largest Occ table and 3 x 8 B/symbol
    for torch.unique over packed H_k windows."""
    occ = max([0] + [(8 * sigma / 32 + 1) if l == 1 else (32 + 4 * sigma) / 32 + 1 for l in layouts])
    per_symbol = 7.5 + max(40.5, 8 + occ, 8 + 24, 8 + 5)
    return int(n * per_symbol) + 2 * GB


# ------------------------------------------------------------------ helpers
def _csr(text, starts, lens):
    """Patterns text[starts[q] : starts[q] + lens[q]] -> (bytes, int64 offsets) on the device."""
    lens = lens.long()
    off = torch.zeros(lens.numel() + 1, dtype=torch.int64, device=text.device)
    off[1:] = torch.cumsum(lens, 0)
    q = torch.repeat_interleave(torch.arange(lens.numel(), device=text.device), lens)
    within = torch.arange(int(off[-1]), device=text.device) - off[:-1][q]
    return text[starts.long()[q] + within], off


def _join(*parts):
    pats = torch.cat([p for p, _ in parts])
    offs, base = [parts[0][1][:1]], 0
    for p, o in parts:
        offs.append(o[1:] + base)
        base += int(o[-1])
    return pats, torch.cat(offs)


def _subset(pats, off, keep):
    """The patterns q with keep[q], in order."""
    lens = (off[1:] - off[:-1])[keep]
    starts = off[:-1][keep]
    return _csr(pats, starts, lens)


def _no_inner_sentinel(pats, off):
    """Keep patterns whose '$' is at most the last symbol: backward search answers those exactly even when the text
    holds '$' elsewhere (a '$' step inside the pattern follows LF across the sentinel rows)."""
    lens = off[1:] - off[:-1]
    P = lens.numel()
    if P == 0:
        return pats, off
    q = torch.repeat_interleave(torch.arange(P, device=off.device), lens)
    pos = torch.arange(pats.numel(), device=off.device) - off[:-1][q]
    inner = (pats == DOLLAR) & (pos < lens[q] - 1)
    bad = torch.zeros(P, dtype=torch.bool, device=off.device)
    bad[q[inner]] = True
    return _subset(pats, off, ~bad)


def _boundary_rows(n):
    """Rows next to every superblock boundary of a level of n bits: k*SUPER_BITS - 1, k*SUPER_BITS, + 1."""
    ks = torch.arange(1, (n - 1) // SUPER_BITS + 1, dtype=torch.int64) * SUPER_BITS
    return torch.cat([ks - 1, ks, ks + 1]).clamp(0, n - 1)


def _marks_of(ssa, n):
    """The mark bit-vector of a sampled-SA blob (rank-block format: 224 payload bits at bytes 4..31 of each 32-byte
    block, little-endian) -> bool[n]."""
    a = int(ssa.plan.off_blocks)
    nblocks = -(-n // BLOCK_BITS)
    blocks = ssa.blob[a:a + 32 * nblocks].view(nblocks, 32)[:, 4:]
    out = torch.empty(nblocks * BLOCK_BITS, dtype=torch.bool, device=ssa.blob.device)
    shifts = torch.arange(8, dtype=torch.uint8, device=ssa.blob.device)
    for g0 in range(0, nblocks, 1 << 20):
        g1 = min(nblocks, g0 + (1 << 20))
        bits = (blocks[g0:g1, :, None] >> shifts) & 1
        out[g0 * BLOCK_BITS:g1 * BLOCK_BITS] = bits.reshape(-1).bool()
    return out[:n]


def _samples_of(ssa):
    a = int(ssa.plan.off_samples)
    return ssa.blob[a:a + 4 * int(ssa.plan.n_samples)].view(torch.int32)


# ------------------------------------------------------------------ the envelope
@pytest.mark.parametrize("case", list(CASES))
def test_index_at_scale(E, case, tmp_path):
    n, make, rate, layouts, unique_sentinel = CASES[case]
    dev = torch.device("cuda", 0)
    torch.cuda.empty_cache()
    sigma_hint = {"eng_max": 97, "bytes255": 256}.get(case, 20)
    need = _peak_bytes(n, sigma_hint, layouts)
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need:
        pytest.skip(f"{case}: needs {need / GB:.1f} GiB of device memory, {free / GB:.1f} GiB free")
    text = make(E, n, dev)
    assert text.numel() == n and int(text[-1]) == DOLLAR
    idx = E.DeviceIndex(text, sa_sample_rate=rate)
    ctx = f"{case}: n={n}, rounds={idx.stats.sa.rounds}, levels={idx.wt.levels}"
    g = torch.Generator(device=dev).manual_seed(n)

    # ---- 1. suffix array, BWT, C[]
    try:
        isa = R.check_suffix_array(text, idx.sa)
    except AssertionError as err:
        raise AssertionError(f"{ctx}: {err}") from None
    assert torch.equal(idx.bwt, R.bwt_of(text, idx.sa)), ctx
    hist = torch.bincount(text.long(), minlength=256)
    Cexcl = torch.cumsum(hist, 0) - hist
    present = hist.nonzero().flatten()
    assert idx.wt.count_table() == {chr(int(c)): int(Cexcl[c]) for c in present}, ctx
    sigma = present.numel()

    # ---- 6. H_k (before the large reference arrays: torch.unique needs ~24 B/symbol)
    ks = (1, 2, 3, 5, 7) + ((12, 20) if case == "dna_max" else ())
    for k in ks:
        want = R.entropy_hk(text, k)
        got = idx.entropy(k)
        assert got == pytest.approx(want, rel=1e-9, abs=1e-12), f"{ctx}: H_{k}"

    # ---- 2. wavelet tree
    bwt = idx.bwt
    for a in range(0, n, 1 << 26):
        b = min(n, a + (1 << 26))
        assert torch.equal(idx.wt.access(torch.arange(a, b, device=dev)), bwt[a:b]), f"{ctx}: access [{a}, {b})"
    groups = R.symbol_positions(bwt)
    rows = torch.cat([torch.tensor([0, n], device=dev), torch.randint(0, n + 1, (4096,), generator=g, device=dev),
                      _boundary_rows(n).to(dev)])
    sym = present.to(torch.uint8).repeat_interleave(rows.numel())
    pos = rows.repeat(sigma)
    assert torch.equal(idx.wt.rank(sym, pos), R.occ_at(bwt, sym, pos, groups)), f"{ctx}: rank"
    for level in range(idx.wt.levels):
        L = idx.wt.level_len(level)
        bits = idx.wt.bv_bits(level, 0, L)
        sb = max(0, (L - 1) // SUPER_BITS - 1) * SUPER_BITS          # one superblock, not the first where there are 2+
        blocks = torch.arange(sb, min(L, sb + SUPER_BITS) + 1, BLOCK_BITS, dtype=torch.int64)
        p = torch.cat([torch.tensor([0, L]), _boundary_rows(L), blocks, blocks - 1]).clamp(0, L).to(dev)
        p = torch.cat([p, torch.randint(0, L + 1, (4096,), generator=g, device=dev)])
        assert torch.equal(idx.wt.bv_rank(level, p), R.bits_rank(bits, p)), f"{ctx}: bv_rank level {level}"
        ones = int(bits.sum())
        assert ones == idx.wt.level_ones(level), ctx
        if ones:
            kk = torch.arange(4096, ones + 1, 4096, dtype=torch.int64)
            kk = torch.cat([torch.tensor([1, ones]), kk - 1, kk, kk + 1]).clamp(1, ones).to(dev)
            kk = torch.cat([kk, torch.randint(1, ones + 1, (4096,), generator=g, device=dev)])
            assert torch.equal(idx.wt.bv_select(level, kk), R.bits_select(bits, kk)), f"{ctx}: bv_select level {level}"
        del bits

    # ---- 3. sampled SA: marks and samples, then locate by LF walks
    sa = idx.sa
    marked = (sa % rate) == 0
    assert torch.equal(_marks_of(idx.ssa, n), marked), f"{ctx}: sampled-SA marks"
    assert torch.equal(_samples_of(idx.ssa), sa[marked] // rate), f"{ctx}: sampled-SA samples"
    mrows = marked.nonzero().flatten()
    qrows = torch.cat([torch.randint(0, n, (1 << 20,), generator=g, device=dev),
                       mrows[:4096], (mrows[:4096] + 1).clamp(max=n - 1), (mrows[:4096] - 1).clamp(min=0),
                       isa[n - 64:].long(), _boundary_rows(n).to(dev)]).to(torch.int32)
    del mrows
    # every row, on every text (also one that holds '$' inside): the position the suffix array holds -- never a
    # wrong position and never none
    want_pos = sa[qrows.long()]
    assert torch.equal(idx.locate_rows(qrows, use_samples=True), want_pos), f"{ctx}: LF-walk locate (tree)"
    del marked

    # ---- 4. count
    body = text[: n - 1]
    letters = present[present != DOLLAR].to(torch.uint8)
    pats, off = E.gen_patterns(n % 1000, 1 << 16, body, letters)
    tail = _csr(text, torch.arange(n - 64, n, device=dev), torch.arange(64, 0, -1, device=dev))
    brow = _boundary_rows(n).to(dev)
    bstart = sa[brow].long()
    across = _csr(text, bstart, (n - bstart).clamp(max=64))
    absent = (torch.randint(0, 256, (256 * 12,), generator=g, device=dev).to(torch.uint8),
              torch.arange(0, 257 * 12, 12, device=dev))
    empty = (torch.zeros(0, dtype=torch.uint8, device=dev), torch.zeros(2, dtype=torch.int64, device=dev))
    pats, off = _no_inner_sentinel(*_join((pats, off), tail, across, absent, empty))
    lo, hi = R.sa_range(text, sa, pats, off)
    for use_kmer in (False, True):
        got = idx.count_batch(pats, off, use_kmer_table=use_kmer, use_occ_table=False)
        assert torch.equal(got[0], lo) and torch.equal(got[1], hi), f"{ctx}: count, kmer table {use_kmer}"
    if case == "dna_max":       # a batch of OCC_MIN_BATCH patterns builds its own Occ table
        P = E.DeviceIndex.OCC_MIN_BATCH
        p2, o2 = E.gen_patterns(5, P, body, letters)
        l2, h2 = R.sa_range(text, sa, p2, o2)
        got = idx.count_batch(p2, o2)
        assert idx._occ is not None and torch.equal(got[0], l2) and torch.equal(got[1], h2), f"{ctx}: count at 2^20"
        idx._occ = None
        del p2, o2, l2, h2
    # locate of the patterns: LF walks == the suffix array, on every pattern with at most 1024 occurrences and on the
    # present pattern with the fewest (a pattern of all_a occurs ~n times, of mississippi_inner >= n/12; the rows of
    # such ranges are covered by the row-level locate above)
    cnt = torch.where(lo >= 0, hi - lo + 1, torch.zeros_like(lo))
    few = cnt <= 1024
    few[torch.where(cnt > 0, cnt, torch.full_like(cnt, n + 1)).argmin()] = True
    lp, lo_ = _subset(pats, off, few)
    o1, p1 = idx.locate_batch(lp, lo_, use_samples=False)
    o2, p2 = idx.locate_batch(lp, lo_, use_samples=True)
    located = f"{ctx}: locate_batch of {int(few.sum())} of {few.numel()} patterns, {int(o1[-1])} positions"
    assert int(o1[-1]) > 0 and torch.equal(o1, o2) and torch.equal(p1, p2), located
    assert torch.equal(o1[1:] - o1[:-1], cnt[few]), located
    first = torch.repeat_interleave(lo[few], cnt[few])             # the rows of every located pattern, in order
    first = first + torch.arange(first.numel(), device=dev) - torch.repeat_interleave(o1[:-1], cnt[few])
    assert torch.equal(p1, sa[first]), located
    del first

    # ---- 5. extract
    S = -(-n // rate)
    isa_s = idx.isa_samples()
    assert torch.equal(isa_s[:S], isa[torch.arange(S, device=dev) * rate]) and int(isa_s[S]) == int(isa_s[0]), ctx
    inv = R.lf_invertible(bwt, isa)
    assert idx.invertible == inv and inv == unique_sentinel, ctx
    R_ = 100_000
    b = torch.randint(0, n + 1, (R_,), generator=g, device=dev)
    e = (b + torch.randint(0, 300, (R_,), generator=g, device=dev)).clamp(max=n)
    extra = torch.tensor([[0, 0], [n, n], [n - 1, n], [n - 300, n], [rate - 1, rate + 1], [7, 8], [0, 1]], device=dev)
    b, e = torch.cat([b, extra[:, 0]]), torch.cat([e, extra[:, 1]])
    if not inv:
        with pytest.raises(ValueError, match="sentinel"):
            idx.extract_batch(b, e)
    else:
        want_off = torch.zeros(b.numel() + 1, dtype=torch.int64, device=dev)
        want_off[1:] = torch.cumsum(e - b, 0)
        want = _csr(text, b, e - b)[0]
        assert torch.equal(idx.extract(0, n, use_occ_table=False), text), f"{ctx}: whole text"
        o, out = idx.extract_batch(b, e, use_occ_table=False)
        assert torch.equal(o, want_off) and torch.equal(out, want), f"{ctx}: extract ranges"

    # ---- Occ tables: count, locate and extract again with LF / rank from the table
    del groups
    for layout in layouts:
        idx.build_occ_table(5, layout=layout)
        got = idx.count_batch(pats, off, use_kmer_table=True, use_occ_table=True)
        assert torch.equal(got[0], lo) and torch.equal(got[1], hi), f"{ctx}: count on Occ layout {layout}"
        assert torch.equal(idx.locate_rows(qrows, use_samples=True), want_pos), f"{ctx}: locate on Occ layout {layout}"
        if inv:
            assert torch.equal(idx.extract(0, n, use_occ_table=True), text), f"{ctx}: whole text, Occ layout {layout}"
            o, out = idx.extract_batch(b, e, use_occ_table=True)
            assert torch.equal(out, want), f"{ctx}: extract ranges, Occ layout {layout}"
        idx._occ = None
        torch.cuda.empty_cache()

    # ---- sample rate 1 at dna_max: n samples, the mark look-back at its widest
    if case == "dna_max":
        idx.ssa, idx._isa, idx._invertible = E.build_sampled_sa(sa, 1), None, None
        assert bool(_marks_of(idx.ssa, n).all()) and torch.equal(_samples_of(idx.ssa), sa), f"{ctx}: rate 1"
        assert torch.equal(idx.locate_rows(qrows, use_samples=True), sa[qrows.long()]), f"{ctx}: locate at rate 1"
        assert torch.equal(idx.isa_samples()[:n], isa), f"{ctx}: isa samples at rate 1"
        assert torch.equal(idx.extract(n - 1000, n), text[n - 1000:]), ctx
        idx.ssa, idx._isa, idx._invertible = E.build_sampled_sa(sa, rate), None, None

    # ---- 7. compressed save / load
    if case in ("dna_max", "eng_max", "all_a_max"):
        path = str(tmp_path / f"{case}.npz")
        idx.save(path, compressed=True)
        back = E.DeviceIndex.load(path, dev)
        os.remove(path)
        a0 = int(idx.wt.plan.off_blocks[0])
        assert back.wt.blob.numel() == idx.wt.blob.numel() and torch.equal(back.wt.blob[a0:], idx.wt.blob[a0:]), \
            f"{ctx}: compressed round trip"
        got = back.count_batch(pats, off, use_kmer_table=False)
        assert torch.equal(got[0], lo) and torch.equal(got[1], hi), f"{ctx}: count on the loaded index"
        assert torch.equal(back.locate_rows(qrows, use_samples=True), want_pos), f"{ctx}: locate on the loaded index"
        del back
    del idx, text, isa, sa, bwt
    torch.cuda.empty_cache()


def test_one_symbol_past_the_limit_is_refused_before_any_kernel(E):
    """2^30 - 1 symbols: DeviceIndex, suffix_array and suffix_array_bwt raise ERANGE; nothing is launched."""
    from hkcsa import _lib
    big = torch.empty(MAX_N + 1, dtype=torch.uint8, device="cuda")
    before = _lib.load().hkcsa_launch_count()
    for fn in (E.DeviceIndex, E.suffix_array, E.suffix_array_bwt):
        with pytest.raises(_lib.HkcsaError) as e:
            fn(big)
        assert e.value.code == _lib.ERANGE
    assert _lib.load().hkcsa_launch_count() == before
