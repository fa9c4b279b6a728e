"""LCP (csrc/lcp.cu): the LCP and PLCP arrays built on the device from the suffix array, against Kasai's algorithm
(tests/lcp_reference.py); the irreducible statistics; Sadakane's 2n-bit encoding and LCP queries on the compressed index
(DeviceIndex.lcp_rows, CompressedSuffixArray(..., lcp=True).lcp).  The argument checks of the C entry points run
without a GPU; everything else is marked gpu."""
import ctypes as C
import math

import numpy as np
import pytest

from lcp_reference import lcp_kasai
from oracle import oracle as O

gpu = pytest.mark.gpu

MAX_N = (1 << 30) - 2


# ------------------------------------------------------------------ texts
def _fib(n):
    a, b = "a", "ab"
    while len(b) < n:
        a, b = b, b + a
    return b[:n]


def _runs(n, seed=5):
    rng = np.random.RandomState(seed)
    out, sym = [], b"xyzw"
    while sum(map(len, out)) < n:
        out.append(bytes([sym[rng.randint(4)]]) * int(rng.randint(1, 200)))
    return b"".join(out)[:n]


def _all_bytes(n, seed=6):
    rng = np.random.RandomState(seed)
    body = rng.randint(0, 256, size=n).astype(np.uint8)
    body[:256] = np.arange(256, dtype=np.uint8)
    return body.tobytes()


def _golden_texts():
    from conftest import Golden, golden_case_names
    g = Golden()
    return {f"golden_{k}": (lambda k=k: g.text(k)) for k in golden_case_names()}


SMALL = {
    "dollar": lambda: b"$",
    "a_dollar": lambda: b"a$",
    "a777": lambda: b"a" * 777 + b"$",
    "dna_300k": lambda: O.gen_text(O.DNA4, 43, 300_000).tobytes() + b"$",
    "eng_300k": lambda: O.gen_text(O.ENG96, 42, 300_000).tobytes() + b"$",
    "fib_1e4": lambda: _fib(10_000).encode() + b"$",
    "fib_1e6": lambda: _fib(1_000_000).encode() + b"$",
    "runs": lambda: _runs(30_000) + b"$",
    "mississippi_x40": lambda: b"mississippi$" * 40 + b"$",
    "ab$ab$": lambda: b"ab$ab$",
    "all_256": lambda: _all_bytes(50_000),
    "no_sentinel": lambda: O.gen_text(O.ENG96, 9, 20_000).tobytes(),
    "binary_1e6": lambda: np.random.RandomState(8).randint(0, 2, 1_000_000).astype(np.uint8).tobytes(),
}
SMALL.update(_golden_texts())


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _irreducible(t: np.ndarray, sa: np.ndarray, plcp: np.ndarray):
    """(count, sum of values) of the irreducible positions: i == 0, i == SA[0], Phi[i] == 0 or t[i-1] != t[Phi[i]-1]."""
    n = len(t)
    if n == 0:
        return 0, 0
    phi = np.zeros(n, dtype=np.int64)
    phi[sa[1:].astype(np.int64)] = sa[:-1]
    i = np.arange(n, dtype=np.int64)
    irr = (i == 0) | (phi == 0) | (t[np.maximum(i - 1, 0)] != t[np.maximum(phi - 1, 0)])
    irr[int(sa[0])] = True
    return int(irr.sum()), int(plcp[irr].astype(np.int64).sum())


def _check_against_kasai(E, text_t, h_text, sa_t, *, stats_check=True):
    """LCP, PLCP and the statistics of the device build against Kasai; returns (lcp, plcp) host uint32 arrays."""
    h_sa = sa_t.cpu().numpy().astype(np.uint32)
    want = lcp_kasai(h_text, h_sa)
    st = []
    lcp, plcp = E.lcp_arrays(text_t, sa_t, lcp=True, plcp=True, stats=st)
    got_lcp = lcp.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_lcp, want), f"LCP differs at row {int(np.flatnonzero(got_lcp != want)[0])}"
    got_plcp = plcp.cpu().numpy().view(np.uint32)
    want_plcp = np.empty_like(want)
    want_plcp[h_sa] = want
    assert np.array_equal(got_plcp, want_plcp)
    if stats_check:
        assert st == list(_irreducible(h_text, h_sa, want_plcp))
    return want, want_plcp, st


@gpu
@pytest.mark.parametrize("name", sorted(SMALL))
def test_lcp_and_plcp_match_kasai(E, name):
    t = SMALL[name]()
    h = np.frombuffer(t, dtype=np.uint8).copy()
    d = E.to_device_u8(t)
    sa = E.suffix_array(d)
    want, _, st = _check_against_kasai(E, d, h, sa)
    # one output at a time gives the same arrays; without stats the call does not wait
    lcp_only, none = E.lcp_arrays(d, sa, lcp=True)
    assert none is None and np.array_equal(lcp_only.cpu().numpy().view(np.uint32), want)
    if name == "fib_1e6":                                       # the work bound of the irreducible compares
        n = len(t)
        assert 0 < st[1] <= 2 * n * math.log2(n)


@gpu
def test_empty_and_one_symbol(E):
    import torch
    L = E._lib.load()
    h = (C.c_uint64 * 2)(7, 7)
    assert L.hkcsa_lcp_build(None, 0, None, None, None, None, 0, h, None) == 0
    assert list(h) == [0, 0]
    d = E.to_device_u8(b"x")
    sa = E.suffix_array(d)
    st = []
    lcp, plcp = E.lcp_arrays(d, sa, lcp=True, plcp=True, stats=st)
    assert lcp.tolist() == [0] and plcp.tolist() == [0] and st == [1, 0]
    bits = torch.full((2,), 7, dtype=torch.uint8, device=d.device)
    assert L.hkcsa_plcp_bits(plcp.data_ptr(), 1, bits.data_ptr(), None) == 0
    assert bits.tolist() == [1, 0]


def test_argument_checks_without_gpu():
    from hkcsa import _lib
    L = _lib.load()
    fake = 256
    need = L.hkcsa_lcp_scratch_bytes(1000)
    assert need >= 4 * 1000
    assert L.hkcsa_lcp_scratch_bytes(MAX_N) <= 5 * MAX_N + (1 << 24)
    assert L.hkcsa_lcp_build(fake, MAX_N + 1, fake, fake, fake, fake, 1 << 40, None, None) == _lib.ERANGE
    assert L.hkcsa_lcp_build(None, 1000, fake, fake, None, fake, need, None, None) == _lib.EINVAL
    assert L.hkcsa_lcp_build(fake, 1000, None, fake, None, fake, need, None, None) == _lib.EINVAL
    assert L.hkcsa_lcp_build(fake, 1000, fake, None, None, fake, need, None, None) == _lib.EINVAL
    assert L.hkcsa_lcp_build(fake, 1000, fake, fake, None, None, need, None, None) == _lib.EINVAL
    assert L.hkcsa_lcp_build(fake, 1000, fake, fake, fake, fake, need - 1, None, None) == _lib.ESCRATCH
    assert L.hkcsa_plcp_bits(fake, MAX_N + 1, fake, None) == _lib.ERANGE
    assert L.hkcsa_plcp_bits(None, 10, fake, None) == _lib.EINVAL
    assert L.hkcsa_plcp_bits(fake, 10, None, None) == _lib.EINVAL
    assert L.hkcsa_plcp_bits(None, 0, None, None) == _lib.OK


# ------------------------------------------------------------------ full size
def _mississippi(n):
    return (b"mississippi$" * (n // 12 + 1))[:n]


FULL = {
    "C2_dna_100MB": lambda E: _gen(E, 1, 43, 100_000_000, sentinel=True),
    "C3_eng_200MB": lambda E: _gen(E, 0, 42, 200_000_000, sentinel=True),
    "dna_max_n": lambda E: _gen(E, 1, 43, MAX_N - 1, sentinel=True),
    "mississippi_max_n": lambda E: E.to_device_u8(_mississippi(MAX_N)),
    "all_a_max_n": lambda E: _all_a(E, MAX_N),
}


def _gen(E, kind, seed, n, sentinel):
    import torch
    t = E.gen_text(kind, seed, n)
    return torch.cat([t, torch.tensor([0x24], dtype=torch.uint8, device=t.device)]) if sentinel else t


def _all_a(E, n):
    import torch
    return torch.full((n,), ord("a"), dtype=torch.uint8, device=torch.device("cuda", 0))


@gpu
@pytest.mark.parametrize("name", list(FULL))
def test_full_size_against_kasai(E, name):
    import torch
    from device_reference import check_suffix_array
    text = FULL[name](E)
    n = text.numel()
    sa = E.suffix_array(text)
    check_suffix_array(text, sa)
    torch.cuda.empty_cache()
    h_text = text.cpu().numpy()
    want, _, st = _check_against_kasai(E, text, h_text, sa, stats_check=n <= 200_000_001)
    if name == "all_a_max_n":       # irreducible: SA[0] = n - 1 (value 0) and 0, whose pair (0, 1) runs n - 1
        assert int(want.max()) == n - 1 and st[0] == 2
    if name == "mississippi_max_n":
        assert int(want.max()) >= n - 13


# ------------------------------------------------------------------ (B) the 2n-bit encoding and queries
def _decoded_plcp(idx):
    import torch
    return idx._plcp_decode(torch.arange(idx.n, dtype=torch.int64, device=idx.device))


def _check_encoding(E, text_t, rate, rows=None):
    import torch
    idx = E.DeviceIndex(text_t, sa_sample_rate=rate)
    plcp = idx.plcp()
    lcp = idx.lcp()
    idx.build_lcp_bits()
    assert torch.equal(_decoded_plcp(idx), plcp.to(torch.int64))
    n = idx.n
    if rows is None:
        rows = torch.arange(n, dtype=torch.int32, device=idx.device)
    want = lcp[rows.long()]
    assert torch.equal(idx.lcp_rows(rows, use_samples=False), want)             # locate through the full SA
    assert torch.equal(idx.lcp_rows(rows, use_samples=True), want)              # through the sampled SA
    idx.sa, idx.text = None, None                                                # what CompressedSuffixArray drops
    assert torch.equal(idx.lcp_rows(rows), want)
    with pytest.raises(ValueError, match="no longer holds"):
        idx.lcp()
    with pytest.raises(ValueError, match="no longer holds"):
        idx.plcp()
    return idx


@gpu
@pytest.mark.parametrize("name", ["a777", "dna_300k", "eng_300k", "fib_1e4", "runs", "all_256", "binary_1e6"])
def test_encoding_and_lcp_rows_small(E, name):
    _check_encoding(E, E.to_device_u8(SMALL[name]()), rate=8)


@gpu
def test_encoding_and_lcp_rows_c2(E):
    import torch
    text = _gen(E, 1, 43, 100_000_000, sentinel=True)
    rows = torch.from_numpy(np.random.RandomState(3).randint(0, text.numel(), 100_000).astype(np.int32)).cuda()
    idx = _check_encoding(E, text, rate=32, rows=rows)
    assert len(idx._lcp_bits) == 1


@gpu
def test_encoding_in_two_pieces(E):
    import torch
    n = (1 << 29) + 4097                         # 2n bits > HKCSA_MAX_N: H is kept as two bit vectors
    text = _gen(E, 1, 5, n - 1, sentinel=True)
    rows = torch.from_numpy(np.random.RandomState(4).randint(0, n, 100_000).astype(np.int32)).cuda()
    idx = _check_encoding(E, text, rate=32, rows=rows)
    assert len(idx._lcp_bits) == 2 and idx._lcp_bits[0].n == MAX_N


@gpu
def test_refusals_of_indexes_without_text_or_sa(E, tmp_path):
    import torch
    t = E.to_device_u8(b"banana$")
    for kw in ({"keep_text": False}, {"keep_sa": False, "sa_sample_rate": 2}):
        idx = E.DeviceIndex(t, **kw)
        for call in (idx.lcp, idx.plcp, idx.build_lcp_bits):
            with pytest.raises(ValueError, match="no longer holds"):
                call()
    idx = E.DeviceIndex(t, sa_sample_rate=2)
    with pytest.raises(ValueError, match="build_lcp_bits"):
        idx.lcp_rows(torch.zeros(1, dtype=torch.int32, device=t.device))
    path = str(tmp_path / "i.npz")
    idx.save(path)
    loaded = E.DeviceIndex.load(path)
    with pytest.raises(ValueError, match="no longer holds"):
        loaded.lcp()


def _csa_expected(text):
    """LCP of text + '$' by direct comparison (str: code points, bytes: byte values)."""
    s = text + ("$" if isinstance(text, str) else b"$")
    seq = [ord(c) for c in s] if isinstance(s, str) else list(s)
    sa = sorted(range(len(seq)), key=lambda i: seq[i:])
    out = [0]
    for r in range(1, len(sa)):
        a, b = seq[sa[r - 1]:], seq[sa[r]:]
        h = 0
        while h < min(len(a), len(b)) and a[h] == b[h]:
            h += 1
        out.append(h)
    return np.array(out, dtype=np.int64)


CSA_TEXTS = {
    "ascii": "abracadabra alakazam " * 30,
    "latin1": "caf\xe9 na\xefve \xfcber " * 40,
    "recoded": "αβγ ☃ αβ " * 40,
    "bytes": O.gen_text(O.DNA4, 2, 3000).tobytes(),
    "holds_dollar": "mississippi$" * 40,
}


@gpu
@pytest.mark.parametrize("name", list(CSA_TEXTS))
def test_csa_lcp(cuda, name, tmp_path):
    from csa.csa import CompressedSuffixArray
    text = CSA_TEXTS[name]
    want = _csa_expected(text)
    csa = CompressedSuffixArray(text, lcp=True)
    n = csa.n
    assert np.array_equal(csa.lcp(range(n)), want)
    assert csa.lcp(5).tolist() == [want[5]]
    rows = np.random.RandomState(1).randint(0, n, 200)
    assert np.array_equal(csa.lcp(rows), want[rows])
    rep = csa.space_report()
    assert rep["lcp_bits_per_symbol"] > 0
    with pytest.raises(ValueError):
        csa.lcp([n])
    plain = CompressedSuffixArray(text)
    assert "lcp_bits_per_symbol" not in plain.space_report()
    assert csa.index_bytes() > plain.index_bytes()
    with pytest.raises(ValueError, match="lcp=True"):
        plain.lcp(0)
    if name != "holds_dollar":
        path = str(tmp_path / "c.npz")
        csa.save(path)
        loaded = CompressedSuffixArray.load(path)
        with pytest.raises(ValueError, match="load"):
            loaded.lcp(0)


@gpu
def test_enhanced_fm_index_lcp_array(cuda):
    from csa.enhanced_fm_index import EnhancedFMIndex
    text = "mississippi" * 20
    fm = EnhancedFMIndex(text)
    want = _csa_expected(text)
    assert fm.lcp_array == want.tolist()
    assert fm.lcp_array is fm.lcp_array
