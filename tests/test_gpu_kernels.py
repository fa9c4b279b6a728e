"""GPU parity tests, kernel by kernel, through the C-ABI (hkcsa.engine -> libhkcsa.so)
against the CPU oracle and the golden fixtures frozen from the reference."""
import numpy as np
import torch
import pytest

from conftest import golden_case_names
from oracle import oracle as O

pytestmark = pytest.mark.gpu

CASES = golden_case_names()


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def dev(E, data):
    return E.to_device_u8(data)


def host(t):
    return t.cpu().numpy()


# ------------------------------------------------------------------ workload generators
@pytest.mark.parametrize("kind,seed,n", [(0, 42, 200_001), (1, 43, 200_001), (0, 7, 1), (1, 9, 65536), (0, 42, 65537)])
def test_textgen_matches_oracle(E, kind, seed, n):
    got = host(E.gen_text(kind, seed, n))
    assert np.array_equal(got, O.gen_text(kind, seed, n))


def test_patterns_match_oracle(E):
    import torch
    text = O.gen_text(O.ENG96, 42, 300_000)
    d_text = dev(E, text)
    alpha = np.unique(text)
    pats, off = E.gen_patterns(44, 5000, d_text, torch.from_numpy(alpha).cuda())
    w_p, w_o = O.gen_patterns(44, 5000, text)
    assert np.array_equal(host(off), w_o)
    assert np.array_equal(host(pats), w_p)


# ------------------------------------------------------------------ radix sort primitive
@pytest.mark.parametrize("n", [1, 2, 31, 100, 4095, 4096, 4097, 100_000, 1_000_003])
@pytest.mark.parametrize("bits", [8, 20, 64])
def test_radix_sort_pairs(E, n, bits):
    import torch
    rng = np.random.RandomState(n % 1000 + bits)
    keys = rng.randint(0, 2 ** 63, size=n, dtype=np.int64).astype(np.uint64) * 2 + rng.randint(0, 2, size=n).astype(np.uint64)
    if bits < 64:
        keys &= np.uint64((1 << bits) - 1)
    vals = np.arange(n, dtype=np.int32)
    dk = torch.from_numpy(keys.view(np.int64)).cuda()
    dv = torch.from_numpy(vals).cuda()
    E.sort_pairs_u64(dk, dv, bits)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(host(dk).view(np.uint64), keys[order])
    assert np.array_equal(host(dv), vals[order])          # stability: equal keys keep input order


def test_radix_sort_few_distinct_keys(E):
    import torch
    n = 300_000
    rng = np.random.RandomState(5)
    keys = (rng.randint(0, 3, size=n).astype(np.uint64) << np.uint64(40)) | rng.randint(0, 2, size=n).astype(np.uint64)
    dk = torch.from_numpy(keys.view(np.int64)).cuda()
    dv = torch.arange(n, dtype=torch.int32, device="cuda")
    E.sort_pairs_u64(dk, dv, 48)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(host(dk).view(np.uint64), keys[order])
    assert np.array_equal(host(dv), order.astype(np.int32))


# ------------------------------------------------------------------ K1 / K2 against the reference's own outputs
@pytest.mark.parametrize("name", CASES)
def test_sa_bwt_golden(E, golden, name):
    text = golden.text(name)
    d_text = dev(E, text)
    sa = E.suffix_array(d_text)
    assert np.array_equal(host(sa).astype(np.uint32), golden.get(f"{name}/sa"))
    got = E.bwt(d_text, sa)
    assert host(got).tobytes() == golden.get(f"{name}/bwt").tobytes()
    if golden.has(f"{name}/fm/sa"):
        d2 = dev(E, text + b"$")
        sa2 = E.suffix_array(d2)
        assert np.array_equal(host(sa2).astype(np.uint32), golden.get(f"{name}/fm/sa"))
        assert host(E.bwt(d2, sa2)).tobytes() == golden.get(f"{name}/fm/bwt").tobytes()


def _texts():
    rng = np.random.RandomState(2024)
    yield "all_a_5000", b"a" * 5000
    yield "ab_period", b"ab" * 4000
    yield "abc_period_tail", b"abc" * 3000 + b"ab"
    yield "fib", _fib(16)
    yield "rand2_100k", bytes(rng.choice(np.frombuffer(b"xy", dtype=np.uint8), 100_000))
    yield "rand256_50k", bytes(rng.randint(0, 256, 50_000).astype(np.uint8))
    yield "runs", b"".join(bytes([65 + (i % 3)]) * int(rng.randint(1, 400)) for i in range(300))
    yield "eng_300k", O.gen_text(O.ENG96, 42, 300_000).tobytes()
    yield "dna_300k", O.gen_text(O.DNA4, 43, 300_000).tobytes()
    yield "dna_1m_dollar", O.gen_text(O.DNA4, 43, 1 << 20).tobytes() + b"$"
    yield "eng_1m_dollar", O.gen_text(O.ENG96, 42, 1 << 20).tobytes() + b"$"
    yield "repeat_block", O.gen_text(O.ENG96, 1, 5000).tobytes() * 20


def _fib(k):
    a, b = b"a", b"ab"
    for _ in range(k):
        a, b = b, b + a
    return b


TEXTS = dict(_texts())


@pytest.mark.parametrize("name", list(TEXTS))
def test_sa_bwt_oracle(E, name):
    text = TEXTS[name]
    d_text = dev(E, text)
    st = E.SaStats()
    sa = E.suffix_array(d_text, st)
    want = O.build_suffix_array(text)
    got = host(sa).astype(np.uint32)
    assert np.array_equal(got, want), f"first mismatch at {np.flatnonzero(got != want)[:5]}"
    assert st.rounds >= 1
    assert host(E.bwt(d_text, sa)).tobytes() == O.bwt_transform(text, want).tobytes()


@pytest.mark.parametrize("env", [{}, pytest.param({"HKCSA_BITS0": "56"}, id="bits0_56"), {"HKCSA_BITS0": "24"},
                                 {"HKCSA_BITS0": "56", "HKCSA_NO_GROUP_ROUND": "1"},
                                 pytest.param({"HKCSA_GRAM": "0", "HKCSA_BITS0": "56"}, id="gram0_bits0_56")])
@pytest.mark.parametrize("name", list(TEXTS))
def test_sa_bwt_one_call(E, name, env, monkeypatch):
    """hkcsa_sa_bwt_build: the BWT symbol rides in the top byte of the round-0 key (keys of at most 56 bits) or the
    gather runs after the build (64-bit keys, unless HKCSA_BITS0 trims them to 56); narrow keys leave many suffixes to the later
    rounds, whose slots get their BWT rows rewritten."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    text = TEXTS[name]
    d_text = dev(E, text)
    st = E.SaStats()
    sa, got = E.suffix_array_bwt(d_text, st)
    want = O.build_suffix_array(text)
    assert np.array_equal(host(sa).astype(np.uint32), want)
    assert host(got).tobytes() == O.bwt_transform(text, want).tobytes()
    if env:
        assert st.bwt_carried == 1 and st.key_bits0 <= 56
    else:
        assert st.bwt_carried == (1 if st.key_bits0 <= 56 else 0)


@pytest.mark.parametrize("name", ["dna_300k", "dna_1m_dollar", "rand2_100k", "runs", "fib", "all_a_5000", "ab_period", "eng_300k"])
def test_round0_key_code_over_grams(E, name, monkeypatch):
    """Small alphabets key round 0 with the order-preserving code over k-grams (k >= 4; built on the device from a
    sampled gram histogram), larger ones with the per-symbol code; HKCSA_GRAM=0 forces the latter.  Same suffix array
    either way, and narrow keys (many survivors: the lazy look-ups recompute gram keys from the text) agree too."""
    text = TEXTS[name]
    d_text = dev(E, text)
    want = O.build_suffix_array(text)
    st = E.SaStats()
    sa = E.suffix_array(d_text, st)
    assert np.array_equal(host(sa).astype(np.uint32), want)
    sigma = len(set(text))
    assert (st.gram_k >= 4) == (sigma <= 18), (st.gram_k, sigma)
    monkeypatch.setenv("HKCSA_GRAM", "0")
    st0 = E.SaStats()
    assert np.array_equal(host(E.suffix_array(d_text, st0)).astype(np.uint32), want) and st0.gram_k == 0
    monkeypatch.delenv("HKCSA_GRAM")
    for bits, extra in (("24", {}), ("32", {"HKCSA_NO_GROUP_ROUND": "1"})):
        monkeypatch.setenv("HKCSA_BITS0", bits)
        for k, v in extra.items():
            monkeypatch.setenv(k, v)
        assert np.array_equal(host(E.suffix_array(d_text)).astype(np.uint32), want)


@pytest.mark.parametrize("n", [1, 2, 7, 8, 9, 4095, 4097, 100_003])
def test_sa_bwt_one_call_ragged_sizes(E, n):
    for kind in (O.ENG96, O.DNA4):
        text = O.gen_text(kind, 3 + n % 5, n).tobytes()
        sa, got = E.suffix_array_bwt(dev(E, text))
        want = O.build_suffix_array(text)
        assert np.array_equal(host(sa).astype(np.uint32), want)
        assert host(got).tobytes() == O.bwt_transform(text, want).tobytes()


@pytest.mark.parametrize("rate", [1, 3, 4, 32, 1000])
@pytest.mark.parametrize("n", [1, 31, 224, 14336, 14337, 100_003, 1_000_001])
def test_sampled_sa_one_pass(E, n, rate):
    """Marks and samples of the sampled suffix array from one pass over the suffix array (look-back over tiles of
    14336 rows): samples = SA[j] / rate of the rows with SA[j] % rate == 0, in row order; marks rank-consistent."""
    rng = np.random.RandomState(n % 1000 + rate)
    perm = rng.permutation(n).astype(np.int32)
    ssa = E.build_sampled_sa(torch.from_numpy(perm).cuda(), rate)
    marked = perm % rate == 0
    want = (perm[marked] // rate).astype(np.uint32)
    assert int(ssa.plan.n_samples) == want.size
    blob = host(ssa.blob)
    off = int(ssa.plan.off_samples)
    got = blob[off:off + 4 * want.size].view(np.uint32)
    assert np.array_equal(got, want)
    bits = np.unpackbits(blob[int(ssa.plan.off_blocks):int(ssa.plan.off_super)].reshape(-1, 32)[:, 4:], axis=1,
                         bitorder="little").reshape(-1)[:n]
    assert np.array_equal(bits.astype(bool), marked)


def test_byte_hist(E):
    rng = np.random.RandomState(3)
    for n in (0, 1, 15, 16, 17, 100_003):
        t = rng.randint(0, 256, n).astype(np.uint8)
        h = E.byte_hist(dev(E, t))
        assert np.array_equal(h, np.bincount(t, minlength=256).astype(np.uint64))
    # unaligned view
    t = rng.randint(0, 256, 4099).astype(np.uint8)
    d = dev(E, t)[3:]
    assert np.array_equal(E.byte_hist(d), np.bincount(t[3:], minlength=256).astype(np.uint64))


# ------------------------------------------------------------------ K3
WT_TEXTS = ["banana", "abcd", "abcde", "mississippi", "this is an example text"]


def _wt_check(E, seq: bytes, full=True):
    d = dev(E, seq)
    wt = E.DeviceWaveletTree(d)
    alpha, spine = O.wt_spine(seq)
    assert wt.alphabet == alpha.tobytes()
    # the full tree is ceil(log2 sigma) deep; the reference's left spine floor(log2 sigma)
    assert wt.levels == (int(np.ceil(np.log2(len(alpha)))) if len(alpha) > 1 else 0)
    assert len(spine) <= wt.levels
    cnt, Ct = O.build_count(seq)
    assert wt.count_table() == {chr(c): int(Ct[c]) for c in range(256) if cnt[c]}
    arr = np.frombuffer(seq, dtype=np.uint8)
    for l, bits in enumerate(spine):
        n_l = len(bits)
        assert wt.level_len(l) >= n_l
        got = host(wt.bv_bits(l, 0, n_l))
        assert np.array_equal(got, bits), f"level {l}"
        rs = O.rank_support(bits)
        assert np.array_equal(host(wt.bv_rank_range(l, 0, n_l + 1)).astype(np.uint32), rs)
    # every level: rank/select against a plain prefix sum of the unpacked bits
    rng = np.random.RandomState(11)
    for l in range(wt.levels):
        L = wt.level_len(l)
        bits = host(wt.bv_bits(l, 0, L))
        rs = np.concatenate([[0], np.cumsum(bits, dtype=np.int64)])
        assert wt.level_ones(l) == int(rs[-1])
        pos = np.unique(np.concatenate([rng.randint(0, L + 1, 200), [0, L, max(0, L - 1), min(L, 224), min(L, 223)]]))
        assert np.array_equal(host(wt.bv_rank(l, pos)), rs[pos])
        ks = np.unique(np.concatenate([rng.randint(0, int(rs[-1]) + 2, 200), [0, 1, int(rs[-1]), int(rs[-1]) + 1]]))
        want = np.searchsorted(rs, ks, side="left")
        want = np.where(ks > rs[-1], L, want)
        assert np.array_equal(host(wt.bv_select(l, ks)), want), f"select level {l}"
    if full and len(seq):
        # occ[c][i] for every symbol at random positions, and access == sequence
        pos = np.unique(np.concatenate([rng.randint(0, len(seq) + 1, 400), [0, len(seq)]]))
        for c in np.unique(arr):
            want = np.concatenate([[0], np.cumsum(arr == c)])[pos]
            got = host(wt.rank(np.full(len(pos), c, dtype=np.uint8), pos))
            assert np.array_equal(got, want), f"rank of {c}"
        absent = [c for c in range(256) if c not in set(arr.tolist())][:1]
        for c in absent:
            assert int(host(wt.rank(np.array([c], dtype=np.uint8), np.array([len(seq)])))[0]) == 0
        ap = np.unique(rng.randint(0, len(seq), 2000))
        assert np.array_equal(host(wt.access(ap)), arr[ap])
    return wt


@pytest.mark.parametrize("s", WT_TEXTS)
def test_wavelet_small(E, s):
    _wt_check(E, s.encode())


@pytest.mark.parametrize("name", ["rand256_50k", "eng_300k", "dna_300k", "runs", "rand2_100k", "dna_1m_dollar"])
def test_wavelet_on_bwt(E, name):
    text = TEXTS[name]
    bwt = O.bwt_transform(text, O.build_suffix_array(text)).tobytes()
    _wt_check(E, bwt)


@pytest.mark.parametrize("sigma", [1, 2, 3, 5, 17, 97, 128, 129, 255, 256])
def test_wavelet_alphabet_sizes(E, sigma):
    rng = np.random.RandomState(sigma)
    seq = rng.randint(0, sigma, 30_000).astype(np.uint8)
    seq[:sigma] = np.arange(sigma)          # every symbol occurs
    _wt_check(E, seq.tobytes())


@pytest.mark.parametrize("name", CASES)
def test_wavelet_golden(E, golden, name):
    meta = golden.meta[name]
    if meta["n"] == 0:
        return
    text = golden.text(name)
    wt = E.DeviceWaveletTree(dev(E, text))
    assert wt.levels >= meta["wt_levels"]
    for l in range(meta["wt_levels"]):
        n_l = int(golden.get(f"{name}/wt/{l}/nbits")[0])
        want = np.unpackbits(golden.get(f"{name}/wt/{l}/bits"))[:n_l]
        assert np.array_equal(host(wt.bv_bits(l, 0, n_l)), want)
        if golden.has(f"{name}/wt/{l}/rank_support"):
            assert np.array_equal(host(wt.bv_rank_range(l, 0, n_l + 1)).astype(np.uint32),
                                  golden.get(f"{name}/wt/{l}/rank_support"))
        ones = int(want.sum())
        m = O.golomb_m(ones, n_l)
        g_len = int(golden.get(f"{name}/wt/{l}/golomb_len")[0])
        want_g = np.unpackbits(golden.get(f"{name}/wt/{l}/golomb"))[:g_len]
        assert np.array_equal(host(wt.golomb(l, n_l, m)), want_g), f"golomb level {l}"


def test_golomb_large_m(E):
    seq = (b"a" * 700 + b"b" * 3 + b"a" * 1300 + b"bbbbbbbbbbbbbbbbbbbbbbb" + b"a" * 5000 + b"b") * 7
    wt = E.DeviceWaveletTree(dev(E, seq))
    bits = (np.frombuffer(seq, dtype=np.uint8) == ord("b")).astype(np.uint8)
    for m in (1, 2, 5, 9):
        assert np.array_equal(host(wt.golomb(0, len(bits), m)), O.golomb_encode(bits, m))
    # a prefix that ends inside a run
    for nb in (701, 702, 2004, 2026, 1792, 1793):
        assert np.array_equal(host(wt.golomb(0, nb, 3)), O.golomb_encode(bits[:nb], 3))


# ------------------------------------------------------------------ K4
def _fm_check(E, text: bytes, P=3000, seed=44, sample_rates=(1, 4, 32)):
    import torch
    t = text + b"$"
    idx = E.DeviceIndex(dev(E, t), sa_sample_rate=sample_rates[-1])
    sa = O.build_suffix_array(t)
    assert np.array_equal(host(idx.sa).astype(np.uint32), sa)
    fm = O.FM(O.bwt_transform(t, sa))
    base = np.frombuffer(text, dtype=np.uint8)
    pats, off = O.gen_patterns(seed, P, base, 1, min(64, len(base)))
    # add empty, unseen-symbol, sentinel and whole-text patterns
    extra = [b"", b"\x01", b"$", text[-1:] + b"$", text[:50], t]
    ep = np.frombuffer(b"".join(extra), dtype=np.uint8)
    pats = np.concatenate([pats, ep])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])])
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    lo, hi = idx.count_batch(d_p, d_o)
    w_lo, w_hi = fm.find_range_batch(pats, off)
    assert np.array_equal(host(lo), w_lo)
    assert np.array_equal(host(hi), w_hi)
    # locate through the full SA (EnhancedFMIndex.find order) and through LF walks
    o1, p1 = idx.locate_batch(d_p, d_o, use_samples=False)
    cnt = np.where(w_lo >= 0, w_hi - w_lo + 1, 0)
    assert np.array_equal(host(o1), np.concatenate([[0], np.cumsum(cnt)]))
    want = np.concatenate([sa[l:h + 1] for l, h in zip(w_lo, w_hi) if l >= 0] or [np.zeros(0, np.uint32)])
    assert np.array_equal(host(p1).astype(np.uint32), want)
    for rate in sample_rates:
        idx.ssa = E.build_sampled_sa(idx.sa, rate)
        o2, p2 = idx.locate_batch(d_p, d_o, use_samples=True)
        assert np.array_equal(host(o2), host(o1))
        assert np.array_equal(host(p2), host(p1)), f"sampled locate, rate {rate}"
    return idx


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "rand2_100k", "runs", "all_a_5000", "fib"])
def test_count_locate_oracle(E, name):
    _fm_check(E, TEXTS[name])


def test_count_text_with_low_bytes(E):
    # bytes below '$' make the sentinel non-minimal (SURVEY A.4)
    rng = np.random.RandomState(8)
    text = bytes(rng.choice(np.frombuffer(b" !#ab\n\t", dtype=np.uint8), 20_000))
    _fm_check(E, text, P=1500)


@pytest.mark.parametrize("name", CASES)
def test_count_locate_golden(E, golden, name):
    import torch
    meta = golden.meta[name]
    if "fm_queries" not in meta:
        return
    idx = E.DeviceIndex(dev(E, golden.text(name) + b"$"))
    qs = meta["fm_queries"]
    d_p, d_o = E.pack_patterns([bytes(q["p"]) for q in qs])
    lo, hi = idx.count_batch(d_p, d_o)
    assert host(lo).tolist() == [q["l"] for q in qs]
    assert host(hi).tolist() == [q["r"] for q in qs]
    o, p = idx.locate_batch(d_p, d_o)
    o, p = host(o), host(p)
    for k, q in enumerate(qs):
        found = p[o[k]:o[k + 1]].tolist()
        assert len(found) == q["find_len"] and sum(found) == q["find_sorted_sum"]
        if q["find"] is not None:
            assert found == q["find"]                      # SA order, as the reference returns
    sym = np.array([c for c, _, _ in meta["fm_rank"]], dtype=np.uint8)
    pos = np.array([i for _, i, _ in meta["fm_rank"]], dtype=np.int64)
    assert host(idx.wt.rank(sym, pos)).tolist() == [v for _, _, v in meta["fm_rank"]]


def test_symbol_positions(E):
    for name in ("eng_300k", "rand256_50k", "all_a_5000"):
        seq = TEXTS[name]
        pos, start = E.symbol_positions(dev(E, seq))
        w_pos, w_start = O.symbol_positions(seq)
        assert np.array_equal(start, w_start)
        assert np.array_equal(host(pos).astype(np.uint32), w_pos)


def test_empty_and_tiny(E):
    import torch
    empty = torch.empty(0, dtype=torch.uint8, device="cuda")
    assert E.suffix_array(empty).numel() == 0                    # build_suffix_array("") == []
    assert E.bwt(empty, E.suffix_array(empty)).numel() == 0
    one = dev(E, b"a")
    assert host(E.suffix_array(one)).tolist() == [0]
    wt = E.DeviceWaveletTree(one)
    assert wt.levels == 0 and wt.sigma == 1
    idx = E.DeviceIndex(dev(E, b"$"))
    lo, hi = idx.count_batch(*E.pack_patterns([b"", b"$", b"a"]))
    assert host(lo).tolist() == [0, 0, -1] and host(hi).tolist() == [0, 0, -1]


# ------------------------------------------------------------------ distributed build, ranks emulated on one GPU
def _emulated_build(E, text, parts, wide, ext_rounds_max=None):
    from hkcsa import dist_sa
    n = len(text)
    d_text = dev(E, text)
    bounds = [n * r // parts for r in range(parts + 1)]
    blocks = [d_text[bounds[r]:bounds[r + 1]].clone() for r in range(parts)]
    kw = {} if ext_rounds_max is None else {"ext_rounds_max": ext_rounds_max}
    return dist_sa.emulate_distributed_suffix_array(blocks, wide=wide, **kw)


def _check_slices(slices, text, wide):
    import torch
    want_sa = O.build_suffix_array(text)
    want_bwt = O.bwt_transform(text, want_sa)
    got_sa = np.concatenate([host(sl.sa_int64()) for sl in slices]).astype(np.uint32)
    got_bwt = np.concatenate([host(sl.bwt) for sl in slices])
    off = 0
    for sl in slices:
        assert sl.offset == off and sl.sa.dtype == (torch.int64 if wide else torch.int32)
        off += sl.sa.numel()
    assert off == len(text)
    assert np.array_equal(got_sa, want_sa)
    assert got_bwt.tobytes() == want_bwt.tobytes()


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "runs", "rand256_50k", "dna_1m_dollar", "rand2_100k"])
@pytest.mark.parametrize("parts", [1, 2, 3, 8])
def test_distributed_slices_concatenate_to_the_suffix_array(E, name, parts):
    """hkcsa.dist_sa with the ranks emulated on one GPU (the per-rank program, the fused pack + exchange kernel,
    the sort and the refinement are the ones torchrun executes; peers' buffers are local buffers): the slices in
    rank order must be the oracle's suffix array and BWT.  32-bit ids, and the 64-bit path texts beyond 4 GB take."""
    text = TEXTS[name]
    for wide in (False, True):
        _check_slices(_emulated_build(E, text, parts, wide), text, wide)


@pytest.mark.parametrize("name", ["all_a_5000", "ab_period", "abc_period_tail", "fib", "repeat_block", "runs"])
@pytest.mark.parametrize("parts", [1, 2, 5, 8])
def test_distributed_build_sorts_repetitive_texts(E, name, parts):
    """LCPs in the thousands: the extension rounds give up and rank doubling over the (emulated) peers' ISA blocks
    finishes -- no text is refused."""
    text = TEXTS[name]
    for wide in (False, True):
        slices = _emulated_build(E, text, parts, wide)
        _check_slices(slices, text, wide)
        assert max(sl.dbl_rounds for sl in slices) >= 1


@pytest.mark.parametrize("name", ["eng_300k", "dna_1m_dollar", "runs", "rand256_50k"])
@pytest.mark.parametrize("parts,stride", [(2, 2), (3, 8), (8, 5)])
def test_distributed_build_with_sampled_cut_points(E, name, parts, stride):
    """Cut points from a histogram over every stride-th tile only, region sizes counted exactly under those cuts
    (hkcsa_dsa_bucket_hist_sampled + hkcsa_dsa_dest_counts): what blocks of 16 M positions and more do."""
    from hkcsa import dist_sa
    text = TEXTS[name]
    d_text = dev(E, text)
    n = len(text)
    cuts = [n * r // parts for r in range(parts + 1)]
    blocks = [d_text[cuts[r]:cuts[r + 1]].clone() for r in range(parts)]
    _check_slices(dist_sa.emulate_distributed_suffix_array(blocks, hist_stride=stride), text, False)


def test_distributed_build_reference_benchmark_workload(E):
    """"mississippi$" * 1000 is the default workload of the reference's own benchmark (tests/benchmark.py:110);
    here 20 000 copies over 4 ranks."""
    text = b"mississippi$" * 20_000
    _check_slices(_emulated_build(E, text, 4, False), text, False)


@pytest.mark.parametrize("env", [{}, {"HKCSA_BITS0": "24"}, {"HKCSA_GRAM": "0", "HKCSA_BITS0": "16"}, {"HKCSA_BITS0": "40"}])
@pytest.mark.parametrize("name", list(TEXTS))
def test_sa_bwt_with_element_parallel_group_round(E, name, env, monkeypatch):
    """Round 1 of the single-GPU builder through the element-parallel group kernel and its second launch for the groups
    it marks; narrow round-0 keys (HKCSA_BITS0) leave many groups, big ones included."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    text = TEXTS[name]
    sa, got = E.suffix_array_bwt(dev(E, text), E.SaStats())
    want = O.build_suffix_array(text)
    assert np.array_equal(host(sa).astype(np.uint32), want)
    assert host(got).tobytes() == O.bwt_transform(text, want).tobytes()


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "runs", "rand256_50k", "dna_1m_dollar", "rand2_100k", "fib"])
@pytest.mark.parametrize("parts", [1, 3, 8])
def test_distributed_build_with_element_parallel_group_round(E, name, parts, monkeypatch):
    """The element-parallel group round gives the right slices, 32- and 64-bit ids: groups across CTA boundaries, groups
    of more than 16, windows that tie or reach the end of the text -- marked for the serial second launch; 64-bit ids
    with and without the key extension bits."""
    text = TEXTS[name]
    for env in ({}, {"HKCSA_DSA_NO_XBITS": "1"}):
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            for wide in (False, True):
                _check_slices(_emulated_build(E, text, parts, wide), text, wide)


@pytest.mark.parametrize("ext", [0, 1, 3])
def test_distributed_doubling_from_any_depth(E, ext):
    """Rank doubling may take over after any number of extension rounds (0: straight after round 0): suffixes that
    were unique by then have no ISA entry and are ranked by the search in their owner's slice."""
    for name in ("eng_300k", "dna_300k", "repeat_block"):
        text = TEXTS[name]
        _check_slices(_emulated_build(E, text, 3, False, ext_rounds_max=ext), text, False)
    _check_slices(_emulated_build(E, TEXTS["dna_300k"], 4, True, ext_rounds_max=ext), TEXTS["dna_300k"], True)


def test_distributed_build_ragged_blocks_and_empty_ranks(E):
    from hkcsa import dist_sa
    text = TEXTS["eng_300k"][:100_003]
    d_text = dev(E, text)
    cuts = [0, 1, 1, 70_001, 100_003]                      # a 1-symbol block, an empty block, unaligned starts
    blocks = [d_text[cuts[r]:cuts[r + 1]].clone() for r in range(4)]
    _check_slices(dist_sa.emulate_distributed_suffix_array(blocks), text, False)
    tiny = b"banana"
    _check_slices(_emulated_build(E, tiny, 8, False), tiny, False)      # more ranks than distinct buckets


@pytest.mark.parametrize("n", [50_000, 50_001, 50_002, 50_003, 131_073])
def test_sa_lazy_round_buffers_any_survivor_parity(E, n):
    """The later-round key buffers are carved at an offset that depends on the number of survivors of round 0
    (odd or even): the TMA bulk copies need 16-byte alignment whatever that number is."""
    for kind in (O.ENG96, O.DNA4):
        text = O.gen_text(kind, 11 + n % 7, n).tobytes()
        sa = E.suffix_array(dev(E, text))
        assert np.array_equal(host(sa).astype(np.uint32), O.build_suffix_array(text))


def test_index_save_load_round_trip(E, tmp_path):
    text = TEXTS["eng_300k"] + b"$"
    idx = E.DeviceIndex(dev(E, text), sa_sample_rate=16)
    path = str(tmp_path / "index.npz")
    idx.save(path)
    back = E.DeviceIndex.load(path)
    pats, off = O.gen_patterns(5, 2000, np.frombuffer(TEXTS["eng_300k"], dtype=np.uint8))
    import torch
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    a, b = idx.count_batch(d_p, d_o), back.count_batch(d_p, d_o)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    o1, p1 = idx.locate_batch(d_p, d_o, use_samples=True)
    o2, p2 = back.locate_batch(d_p, d_o)                     # replica has no full SA: LF walks
    assert torch.equal(o1, o2) and torch.equal(p1, p2)


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "runs", "rand256_50k", "all_a_5000", "fib", "rand2_100k"])
def test_rrr_coded_levels_rank_and_round_trip(E, name):
    """csrc/rrr.cu: every wavelet-tree level in the class/offset code -- rank on the coded form equals rank on the
    plain level at block / superblock boundaries and random positions, and decoding gives the level back bit for bit."""
    import torch
    seq = TEXTS[name]
    wt = E.DeviceWaveletTree(dev(E, seq))
    rng = np.random.RandomState(7)
    for level in range(wt.levels):
        n_l = wt.level_len(level)
        vec = E.RrrVector.encode(wt, level)
        assert vec.nbits == n_l and int(vec.plan.ones) == wt.level_ones(level)
        want_bits = host(wt.bv_bits(level, 0, n_l))
        assert np.array_equal(host(vec.bits()), want_bits)
        if n_l > 2000:
            assert np.array_equal(host(vec.bits(959, 1000)), want_bits[959:1959])       # a range across superblocks
        edge = [0, 1, 14, 15, 16, 959, 960, 961, n_l - 1, n_l, n_l + 5]
        pos = np.unique(np.clip(np.concatenate([edge, rng.randint(0, n_l + 1, 3000)]), 0, None)).astype(np.int64)
        want = np.concatenate([[0], np.cumsum(want_bits, dtype=np.int64)])[np.minimum(pos, n_l)]
        assert np.array_equal(host(vec.rank(pos)), want)
        assert np.array_equal(host(wt.bv_rank(level, np.minimum(pos, n_l))), want)
    # a sparse and a dense stand-alone vector: the code is far below / slightly above one bit per bit
    for p_one, lo, hi in ((0.01, 0.3, 0.4), (0.5, 1.0, 1.25)):       # 4 / 15 class bits + 64 / 960 + the offsets
        bits = (rng.random_sample(200_003) < p_one).astype(np.uint8)
        bv = E.DeviceBitVector(torch.from_numpy(bits).cuda())
        vec = E.RrrVector.encode(bv, 0)
        assert np.array_equal(host(vec.bits()), bits)
        assert lo < vec.coded_bits / len(bits) < hi


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "runs", "all_a_5000"])
def test_index_save_compressed_load_round_trip(E, tmp_path, name):
    """save(compressed=True) writes the coded levels; load() decodes them in place and rebuilds the rank directories:
    the restored query blob is bit-identical to the original and answers identically."""
    import os
    import torch
    text = TEXTS[name] + b"$"
    idx = E.DeviceIndex(dev(E, text), sa_sample_rate=16)
    plain, coded = str(tmp_path / "plain.npz"), str(tmp_path / "coded.npz")
    idx.save(plain)
    idx.save(coded, compressed=True)
    back = E.DeviceIndex.load(coded)
    if idx.wt.levels:                       # rank blocks, superblocks and select samples of every level, bit for bit
        lv = int(idx.wt.plan.off_blocks[0])   # (the bytes before them are node tables + alignment padding)
        assert torch.equal(back.wt.blob[lv:], idx.wt.blob[lv:])
    pats, off = O.gen_patterns(5, 2000, np.frombuffer(TEXTS[name], dtype=np.uint8), 1, 30)
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    a, b = idx.count_batch(d_p, d_o), back.count_batch(d_p, d_o)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    o1, p1 = idx.locate_batch(d_p, d_o, use_samples=True)
    o2, p2 = back.locate_batch(d_p, d_o)
    assert torch.equal(o1, o2) and torch.equal(p1, p2)
    sp = idx.space()
    assert sp["coded_level_bits_per_symbol"] > 0 and len(sp["coded_bits_per_level"]) == idx.wt.levels
    if name in ("runs", "all_a_5000"):                       # long runs: far below the raw level bits
        assert sp["coded_level_bits_per_symbol"] < 0.6 * max(sp["raw_level_bits_per_symbol"], 1e-9) or idx.wt.levels == 0


def test_compressed_suffix_array_space_report_next_to_entropy(E):
    """CompressedSuffixArray.space_report(): index bits per symbol next to n*H_k (the reference's README.md:4-11 claim
    'space close to the k-th order entropy' made measurable).  On the order-3 Markov text H_3 << H_0 and the coded
    wavelet tree of the BWT sits between them."""
    from csa.csa import CompressedSuffixArray
    text = O.gen_text(O.ENG96, 42, 300_000).tobytes().decode("latin-1")
    csa = CompressedSuffixArray(text, entropy_orders=(0, 1, 2, 3, 4))
    rep = csa.space_report()
    H = rep["H_k_bits_per_symbol"]
    assert H[0] > H[1] > H[2] > H[3] >= H[4] > 0
    assert rep["n_H_k_bits"][3] == pytest.approx(H[3] * csa.n)
    # the 15-bit class/offset code pays 4/15 + 1/15 bits per level bit on top of the blocks' entropy: on a text this
    # small only the run-heavy levels shrink, the others are kept plain -- never above the raw levels
    assert H[3] * 0.9 < rep["coded_level_bits_per_symbol"] <= rep["raw_level_bits_per_symbol"]
    assert rep["stored_bits_per_level"] == [min(a, b) for a, b in zip(rep["coded_bits_per_level"],
                                                                      [rep["stored_bits_per_level"][l] if l in rep["levels_kept_plain"] else 10 ** 18
                                                                       for l in range(rep["levels"])])]
    assert csa.locate(text[1000:1012]) == sorted(i for i in range(len(text)) if text.startswith(text[1000:1012], i))


@pytest.mark.parametrize("name,parts", [("eng_300k", 3), ("dna_300k", 8), ("rand2_100k", 2), ("dna_1m_dollar", 5), ("runs", 4)])
def test_multi_slice_index_matches_single_index(E, name, parts):
    """hkcsa.dist_sa.MultiSliceIndex (the index a distributed build leaves behind) must answer exactly like the
    single-GPU index: count ranges, and positions from LF walks that hop across slices."""
    import torch
    from hkcsa import dist_sa
    text = TEXTS[name] + (b"" if name.endswith("dollar") else b"$")
    d_text = dev(E, text)
    idx = E.DeviceIndex(d_text, sa_sample_rate=8)
    n = len(text)
    cuts = [n * r // parts for r in range(parts + 1)]
    wide = parts % 2 == 1                         # odd part counts exercise the 64-bit suffix-id path
    slices = [{"bwt": idx.bwt[cuts[r]:cuts[r + 1]].clone(),
               "sa": idx.sa[cuts[r]:cuts[r + 1]].to(torch.int64) if wide else idx.sa[cuts[r]:cuts[r + 1]].clone()}
              for r in range(parts)]
    ms = dist_sa.MultiSliceIndex(n, slices, sa_sample_rate=8)
    base = np.frombuffer(text[:-1], dtype=np.uint8)
    pats, off = O.gen_patterns(9, 3000, base, 1, 40)
    extra = [b"", b"\x01", b"$", text[-2:], text[:30]]
    pats = np.concatenate([pats, np.frombuffer(b"".join(extra), dtype=np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])])
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    lo, hi = idx.count_batch(d_p, d_o)
    mlo, mhi = ms.count_batch(d_p, d_o)
    assert torch.equal(lo, mlo) and torch.equal(hi, mhi)
    o1, p1 = idx.locate_batch(d_p, d_o, use_samples=False)
    o2, p2 = ms.locate_batch(d_p, d_o)
    assert torch.equal(o1, o2) and torch.equal(p1.to(torch.int64), p2)
    # more patterns than the count grid has lanes (148 SMs x 8 CTAs x 256 threads): lanes refill with the next
    # pattern of their warp's chunk
    pats, off = O.gen_patterns(10, 400_000, base, 1, 40)
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    lo, hi = idx.count_batch(d_p, d_o)
    mlo, mhi = ms.count_batch(d_p, d_o)
    assert torch.equal(lo, mlo) and torch.equal(hi, mhi)


def test_property_random_small_texts(E):
    """hypothesis: small texts over tiny alphabets (many repeats, every tail shape) -- SA, BWT, count and locate
    through the C-ABI equal the oracle."""
    import torch
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=150, deadline=None)
    @given(st.binary(min_size=0, max_size=300).map(lambda b: bytes(97 + (x % 3) for x in b)),
           st.binary(min_size=0, max_size=6).map(lambda b: bytes(97 + (x % 3) for x in b)))
    def check(text, pat):
        d = dev(E, text)
        sa = E.suffix_array(d)
        want = O.build_suffix_array(text)
        assert np.array_equal(host(sa).astype(np.uint32), want)
        assert host(E.bwt(d, sa)).tobytes() == O.bwt_transform(text, want).tobytes()
        t = text + b"$"
        idx = E.DeviceIndex(dev(E, t), sa_sample_rate=3)
        sa2 = O.build_suffix_array(t)
        fm = O.FM(O.bwt_transform(t, sa2))
        lo, hi = idx.count_batch(*E.pack_patterns([pat]))
        l, r = fm.find_range(pat)
        assert (int(lo.item()), int(hi.item())) == (l, r)
        o, p = idx.locate_batch(*E.pack_patterns([pat]), use_samples=True)
        assert host(p).tolist() == ([] if l < 0 else sa2[l:r + 1].tolist())

    check()


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "rand2_100k", "runs", "rand256_50k", "all_a_5000"])
def test_kmer_jump_table_gives_identical_ranges(E, name):
    import torch
    text = TEXTS[name] + b"$"
    idx = E.DeviceIndex(dev(E, text))
    base = np.frombuffer(TEXTS[name], dtype=np.uint8)
    pats, off = O.gen_patterns(21, 4000, base, 1, 40)
    extra = [b"", b"\x01", b"$", text[-3:], text[:25], b"\x01" + text[:12], text[:12] + b"\x01"]
    pats = np.concatenate([pats, np.frombuffer(b"".join(extra), dtype=np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])])
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    a = idx.count_batch(d_p, d_o, use_kmer_table=False)
    b = idx.count_batch(d_p, d_o, use_kmer_table=True)
    assert idx._kmer is not None
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    fm = O.FM(O.bwt_transform(text, O.build_suffix_array(text)))
    w_lo, w_hi = fm.find_range_batch(pats, off)
    assert np.array_equal(host(b[0]), w_lo) and np.array_equal(host(b[1]), w_hi)


@pytest.mark.parametrize("shift,layout", [(5, 0), (6, 0), (5, 1)])
@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "rand2_100k", "runs", "rand256_50k", "all_a_5000", "fib"])
def test_occ_table_count_matches_wavelet_count_and_oracle(E, name, shift, layout):
    """hkcsa_count_batch_occ (sampled Occ table, the reference's build_occ kept at every 2^shift-th row) against the
    wavelet-tree count and the oracle's find_range; with and without the k-mer jump table."""
    import torch
    text = TEXTS[name] + b"$"
    idx = E.DeviceIndex(dev(E, text))
    base = np.frombuffer(TEXTS[name], dtype=np.uint8)
    pats, off = O.gen_patterns(23, 4000, base, 1, 48)
    extra = [b"", b"\x01", b"$", text[-3:], text[:25], b"\x01" + text[:12], text[:12] + b"\x01", text[-70:]]
    pats = np.concatenate([pats, np.frombuffer(b"".join(extra), dtype=np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])])
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    a = idx.count_batch(d_p, d_o, use_kmer_table=False)
    idx.ssa = E.build_sampled_sa(idx.sa, 16)
    o_ref, p_ref = idx.locate_batch(d_p, d_o, use_samples=True)     # LF walks on the wavelet tree
    plan, blob = idx.build_occ_table(shift, layout=layout)
    assert plan.rows == (len(text) >> shift) + 1
    o_occ, p_occ = idx.locate_batch(d_p, d_o, use_samples=True)     # LF walks on the Occ table
    assert torch.equal(o_ref, o_occ) and torch.equal(p_ref, p_occ)
    b = idx.count_batch(d_p, d_o, use_kmer_table=False, use_occ_table=True)
    c = idx.count_batch(d_p, d_o, use_kmer_table=True)            # occ table + jump table
    for got in (b, c):
        assert torch.equal(a[0], got[0]) and torch.equal(a[1], got[1])
    fm = O.FM(O.bwt_transform(text, O.build_suffix_array(text)))
    w_lo, w_hi = fm.find_range_batch(pats, off)
    assert np.array_equal(host(b[0]), w_lo) and np.array_equal(host(b[1]), w_hi)
    # the kept rows are the reference's occ[c][r << shift] and the stored symbols are the BWT
    bwt = np.asarray(fm.bwt, dtype=np.uint8)
    syms = sorted(set(text))
    check_rows = (0, 1, plan.rows // 2, plan.rows - 1)
    if layout == 0:
        assert plan.stride % 32 == 0
        rows = host(blob)[:plan.rows * plan.stride].reshape(plan.rows, plan.stride)
        B = 1 << shift
        assert np.array_equal(rows[:, :B].reshape(-1)[:len(text)], bwt)
        counters = rows[:, B:B + 4 * plan.sigma].copy().view(np.uint32)
        for r in check_rows:
            pos = min(r << shift, len(text))
            assert counters[r].tolist() == [int(np.count_nonzero(bwt[:pos] == s)) for s in syms]
    else:       # per symbol: entry[code][r] = (occ[code][32 r], bitmap of the 32 rows holding the symbol); BWT copy at the end
        h = host(blob)
        ent = h[:plan.sigma * plan.stride * 8].copy().view(np.uint32).reshape(plan.sigma, plan.stride, 2)
        assert np.array_equal(h[plan.off_bwt:plan.off_bwt + len(text)], bwt)
        for r in check_rows:
            pos = min(r << 5, len(text))
            assert ent[:, r, 0].tolist() == [int(np.count_nonzero(bwt[:pos] == s)) for s in syms]
            seg = bwt[pos:pos + 32]
            assert ent[:, r, 1].tolist() == [sum(1 << j for j in range(len(seg)) if seg[j] == s) for s in syms]


@pytest.mark.parametrize("n", [8192, 16384, 8191, 8193, 64, 1])
def test_occ_table_at_tile_boundaries(E, n):
    import torch
    rng = np.random.RandomState(n)
    text = bytes(rng.choice(np.frombuffer(b"abc", dtype=np.uint8), n - 1)) + b"$" if n > 1 else b"$"
    idx = E.DeviceIndex(dev(E, text))
    idx.build_occ_table(5, layout=n % 2)
    pats = [text[i:i + 6] for i in range(0, max(1, len(text) - 6), max(1, len(text) // 50))] + [b"", b"$", b"zz"]
    d_p, d_o = E.pack_patterns(pats)
    a = idx.count_batch(d_p, d_o, use_occ_table=False)
    b = idx.count_batch(d_p, d_o, use_occ_table=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("use_occ", [False, True])
def test_count_batch_peers_writes_every_peer_array(E, use_occ):
    """hkcsa_count_batch_peers (the gather fused into the search) with the "peers" being plain buffers on this GPU:
    a slice of the batch searched with out_base lands at its place in every peer array, equal to count_batch."""
    import ctypes as C
    import torch
    text = TEXTS["eng_300k"] + b"$"
    idx = E.DeviceIndex(dev(E, text))
    if use_occ:
        idx.build_occ_table(5, layout=1)
    pats, off = O.gen_patterns(29, 3000, np.frombuffer(TEXTS["eng_300k"], dtype=np.uint8), 1, 40)
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    want_lo, want_hi = idx.count_batch(d_p, d_o, use_kmer_table=False)
    P = 3000
    bufs = [torch.full((2, P), -7, dtype=torch.int64, device="cuda") for _ in range(3)]
    peer_lo = (C.c_uint64 * 3)(*[b.data_ptr() for b in bufs])
    peer_hi = (C.c_uint64 * 3)(*[b.data_ptr() + 8 * P for b in bufs])
    from hkcsa import dist as hdist
    for b0, e0 in ((0, 1100), (1100, 1100), (1100, 3000)):            # three "ranks", one of them with an empty slice
        lp, lo_ = hdist.local_slice(d_p, d_o, b0, e0)
        idx.count_batch_peers(lp, lo_, b0, peer_lo, peer_hi, use_kmer_table=False)
    torch.cuda.synchronize()
    for b in bufs:
        assert torch.equal(b[0], want_lo) and torch.equal(b[1], want_hi)


def test_ranges_push_peers_packs_and_unpacks(E):
    """hkcsa_ranges_push_peers (the result gather as a store kernel) with the "peers" being plain buffers on this
    GPU: slices with odd and even bases, an empty slice and a one-pattern slice land packed at their place in every
    peer array; hkcsa_ranges_unpack gives back count_batch's (lo, hi)."""
    import ctypes as C
    import torch
    from hkcsa import _lib
    L = _lib.load()
    text = TEXTS["eng_300k"] + b"$"
    idx = E.DeviceIndex(dev(E, text))
    pats, off = O.gen_patterns(31, 3001, np.frombuffer(TEXTS["eng_300k"], dtype=np.uint8), 1, 40)
    extra = [b"", b"\x01"]                                  # the whole range (count = n), and a miss
    pats = np.concatenate([pats, np.frombuffer(b"".join(extra), dtype=np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])])
    P = len(off) - 1
    d_p, d_o = torch.from_numpy(pats).cuda(), torch.from_numpy(off).cuda()
    want_lo, want_hi = idx.count_batch(d_p, d_o, use_kmer_table=False)
    bufs = [torch.full((P + 1,), -7, dtype=torch.int64, device="cuda") for _ in range(3)]
    peers = (C.c_uint64 * 3)(*[b.data_ptr() for b in bufs])
    st = torch.cuda.current_stream().cuda_stream
    for b0, e0 in ((0, 1101), (1101, 1101), (1101, 1102), (1102, 2000), (2000, P)):
        lo, hi = want_lo[b0:e0].contiguous(), want_hi[b0:e0].contiguous()
        _lib.check(L.hkcsa_ranges_push_peers(lo.data_ptr(), hi.data_ptr(), e0 - b0, b0, 3, peers, 0, st))
    torch.cuda.synchronize()
    for b in bufs:
        assert int(b[P].item()) == -7                       # nothing stored past the batch
        lo = torch.empty(P, dtype=torch.int64, device="cuda")
        hi = torch.empty_like(lo)
        _lib.check(L.hkcsa_ranges_unpack(b.data_ptr(), P, lo.data_ptr(), hi.data_ptr(), st))
        assert torch.equal(lo, want_lo) and torch.equal(hi, want_hi)
    packed = host(bufs[0][:P]).view(np.uint64)
    assert packed[P - 2] == (np.uint64(len(text)) << np.uint64(32)) and packed[P - 1] == np.uint64(0xFFFFFFFF)


@pytest.mark.parametrize("name", ["eng_300k", "dna_300k", "runs", "fib"])
def test_psi_is_the_inverse_of_lf(E, name):
    """DeviceIndex.psi(): SA[psi[i]] = SA[i] + 1 (mod n) for every row, and psi equals the concatenation of the
    reference's precompute_rank position lists (oracle restatement)."""
    text = TEXTS[name] + b"$"
    idx = E.DeviceIndex(dev(E, text))
    psi = host(idx.psi()).astype(np.int64)
    sa = host(idx.sa).astype(np.int64)
    n = len(text)
    assert np.array_equal(sa[psi], (sa + 1) % n)
    w_pos, _ = O.symbol_positions(host(idx.bwt))
    assert np.array_equal(psi.astype(np.uint32), w_pos)


@pytest.mark.parametrize("mode", ["wt", "occ0_shift5", "occ0_shift6", "occ1"])
@pytest.mark.parametrize("text,rate", [(b"ab$ab$", 6), (b"a$b$a$", 2), (b"mississippi$" * 400 + b"$", 32),
                                       (b"mississippi$" * 40 + b"$", 5), (b"banana$", 3)])
def test_sampled_locate_is_exact_when_the_last_symbol_occurs_earlier(E, text, rate, mode):
    """A text that holds its last symbol elsewhere too (a second '$'): occ alone ranks the row of suffix 0 after the
    other rows holding that symbol, so a plain LF step goes wrong there -- on "mississippi$" * 400 + "$" at rate 32,
    600 of 4801 walks reported a position 12 too far and 3000 none.  The locate kernels take the exact step (row0
    from the inverse samples): every row gives the position its suffix-array entry holds, on the tree and on every
    Occ-table layout, also from an index that keeps no suffix array."""
    n = len(text)
    sa = O.build_suffix_array(text).astype(np.int64)
    idx = E.DeviceIndex(dev(E, text), sa_sample_rate=rate, keep_sa=False)
    if mode != "wt":
        layout, shift = (1, 5) if mode == "occ1" else (0, int(mode[-1]))
        idx.build_occ_table(shift, layout=layout)
    assert idx.row_of_suffix0() == int(np.flatnonzero(sa == 0)[0])
    rows = torch.arange(n, dtype=torch.int32, device="cuda")
    got = idx.locate_rows(rows).cpu().numpy().astype(np.int64)       # no suffix array: the samples are used
    assert np.array_equal(got, sa)
    o, p = idx.locate_batch(*E.pack_patterns([b"ss", b"$", b"i$", b"a"]))
    o, p = o.cpu().numpy(), p.cpu().numpy()
    for k, pat in enumerate([b"ss", b"$", b"i$", b"a"]):
        assert sorted(p[o[k]:o[k + 1]].tolist()) == [m for m in range(n) if text.startswith(pat, m)], pat
