"""The sliced index a distributed build leaves behind (hkcsa.dist_sa.MultiSliceIndex), checked row by row against the
oracle's suffix array: locate by LF walks that hop across slices on every row, count against the oracle's
find_range, and the index built straight from what emulate_distributed_suffix_array returns.  Also the size checks
of the distributed build that refuse a slice beyond one GPU's limit.

Texts that hold their last symbol earlier too ("mississippi$" * k, a second '$', an English-like text whose last
letter recurs) are where a plain LF step goes wrong: occ alone ranks the row of suffix 0 after the other rows
holding that symbol (DESIGN section 3 K4)."""
import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _oracle(text: bytes):
    sa = O.build_suffix_array(text).astype(np.int64)
    return sa, O.bwt_transform(text, sa.astype(np.uint32))


def _ms_from_sa(text, sa, bwt, cuts, rate, wide):
    """A MultiSliceIndex over the oracle's suffix array and BWT cut at `cuts` (empty slices allowed)."""
    from hkcsa import dist_sa
    slices = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        ids = torch.from_numpy(sa[a:b].copy()).cuda()
        slices.append({"bwt": torch.from_numpy(bwt[a:b].copy()).cuda(),
                       "sa": ids if wide else ids.to(torch.int32)})
    return dist_sa.MultiSliceIndex(len(text), slices, sa_sample_rate=rate)


PATTERNS = [b"", b"a", b"b", b"$", b"ab", b"b$", b"$a", b"a$", b"ss", b"i$", b"ssi", b"mis", b"ppi$", b"p", b"x"]


def _check_locate(E, ms, text, sa, bwt, patterns):
    """Every row through locate_rows; count == the oracle's find_range; locate_batch == the SA range of the count."""
    n = len(text)
    assert ms.row0 == int(np.flatnonzero(sa == 0)[0])
    got = ms.locate_rows(torch.arange(n, dtype=torch.int64, device="cuda")).cpu().numpy()
    wrong = int((got != sa).sum())
    missing = int((got == -1).sum())
    assert wrong == 0, f"{wrong} of {n} rows wrong ({missing} without a position)"
    pats, off = E.pack_patterns(patterns)
    lo, hi = ms.count_batch(pats, off)
    w_lo, w_hi = O.FM(bwt).find_range_batch(pats.cpu().numpy(), off.cpu().numpy())
    assert np.array_equal(lo.cpu().numpy(), w_lo) and np.array_equal(hi.cpu().numpy(), w_hi)
    o, p = ms.locate_batch(pats, off)
    o, p = o.cpu().numpy(), p.cpu().numpy()
    for q in range(len(w_lo)):
        want = sa[w_lo[q]:w_hi[q] + 1] if w_lo[q] >= 0 else sa[:0]
        assert np.array_equal(p[o[q]:o[q + 1]], want), patterns[q]


LOCATE_TEXTS = {
    "mississippi_k": b"mississippi$" * 40,                 # the reference benchmark's text: '$' recurs, none extra
    "mississippi_k_dollar": b"mississippi$" * 40 + b"$",
    "ab$ab$": b"ab$ab$",
    "a$b$a$": b"a$b$a$",
    "banana$": b"banana$",                                 # unique sentinel: the plain step
}


@pytest.mark.parametrize("name", list(LOCATE_TEXTS))
@pytest.mark.parametrize("rate", [1, 3, 32])
@pytest.mark.parametrize("parts", [1, 2, 3, 8])
def test_multi_slice_locate_every_row(E, name, rate, parts):
    """locate_rows on all n rows equals the suffix array; 1-8 slices (empty ones on the short texts), 64-bit ids on
    odd slice counts."""
    text = LOCATE_TEXTS[name]
    sa, bwt = _oracle(text)
    n = len(text)
    cuts = [n * r // parts for r in range(parts + 1)]
    ms = _ms_from_sa(text, sa, bwt, cuts, rate, wide=parts % 2 == 1)
    _check_locate(E, ms, text, sa, bwt, PATTERNS + [text[:12], text[-3:]])


@pytest.mark.parametrize("edge", ["first", "last"])
@pytest.mark.parametrize("rate", [3, 32])
def test_multi_slice_locate_with_row0_at_a_slice_edge(E, edge, rate):
    """The row of suffix 0 as the first row of a slice and as the last: c0 and the fix are read in one slice, the
    c0-rows before row0 lie in others."""
    text = b"mississippi$" * 60 + b"$"
    sa, bwt = _oracle(text)
    n = len(text)
    row0 = int(np.flatnonzero(sa == 0)[0])
    cut = row0 if edge == "first" else row0 + 1
    assert 0 < cut < n
    cuts = sorted({0, n // 5, cut, (4 * n) // 5, n})
    ms = _ms_from_sa(text, sa, bwt, cuts, rate, wide=False)
    s = cuts.index(cut)
    assert (ms.starts[s] == row0) if edge == "first" else (ms.starts[s] == row0 + 1)
    _check_locate(E, ms, text, sa, bwt, PATTERNS)


def _texts():
    yield "eng_300k", O.gen_text(O.ENG96, 42, 300_000).tobytes(), 3           # last letter recurs
    yield "dna_1m_dollar", O.gen_text(O.DNA4, 43, 1 << 20).tobytes() + b"$", 5
    yield "mississippi_20000", b"mississippi$" * 20_000, 4
    yield "banana_8_ranks", b"banana", 8                                        # empty slices


DIST_TEXTS = {name: (text, parts) for name, text, parts in _texts()}


@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("name", list(DIST_TEXTS))
def test_multi_slice_index_over_the_distributed_build(E, name, wide):
    """The slices emulate_distributed_suffix_array returns (their BWT and suffix ids, 32- or 64-bit) make the index
    directly: count against the oracle's find_range, locate on every row against the oracle's suffix array."""
    from hkcsa import dist_sa
    text, parts = DIST_TEXTS[name]
    n = len(text)
    d = E.to_device_u8(text)
    bounds = [n * r // parts for r in range(parts + 1)]
    slices = dist_sa.emulate_distributed_suffix_array([d[bounds[r]:bounds[r + 1]].clone() for r in range(parts)],
                                                      wide=wide)
    sa, bwt = _oracle(text)
    assert [sl.offset for sl in slices] == list(np.cumsum([0] + [sl.sa.numel() for sl in slices[:-1]]))
    if name == "banana_8_ranks":
        assert any(sl.sa.numel() == 0 for sl in slices)
    ms = dist_sa.MultiSliceIndex(n, [{"bwt": sl.bwt, "sa": sl.sa} for sl in slices], sa_sample_rate=32)
    pats, off = O.gen_patterns(9, 3000, np.frombuffer(text, dtype=np.uint8), 1, min(40, n))
    extra = [b"", b"\x01", b"$", text[-2:], text[:30], text[-30:]]
    patterns = [pats[off[q]:off[q + 1]].tobytes() for q in range(len(off) - 1)] + extra
    _check_locate(E, ms, text, sa, bwt, patterns)


def test_replicated_sliced_index_carries_the_row_of_suffix_0(E):
    """replicate_sliced_index (one NCCL rank in this process): the all-gathered header brings the row of suffix 0, so
    the replica's walks are exact on a text whose last symbol recurs."""
    import torch.distributed as dist
    from hkcsa import dist_sa
    text = b"mississippi$" * 2_000
    sa, _ = _oracle(text)
    sl, = dist_sa.emulate_distributed_suffix_array([E.to_device_u8(text)])
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        ms = dist_sa.replicate_sliced_index(sl, sa_sample_rate=32)
    finally:
        dist.destroy_process_group()
    assert ms.row0 == int(np.flatnonzero(sa == 0)[0])
    got = ms.locate_rows(torch.arange(len(text), device="cuda")).cpu().numpy()
    assert np.array_equal(got, sa)


# ------------------------------------------------------------------ refusals: a slice beyond one GPU's limit
def test_one_rank_past_the_slice_limit_is_refused_before_the_workspace(E):
    """One emulated rank over 2^30 - 1 symbols: its slice exceeds HKCSA_MAX_N, refused with ERANGE after the
    histograms and before the receive arrays (~20 B/symbol) are allocated."""
    from hkcsa import _lib, dist_sa
    n = _lib.MAX_N + 1
    block = E.gen_text(E.ENG96, 5, n)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with pytest.raises(_lib.HkcsaError) as e:
        dist_sa.emulate_distributed_suffix_array([block])
    assert e.value.code == _lib.ERANGE and "exceeds" in str(e.value)
    assert torch.cuda.max_memory_allocated() - base < 3 * n             # the replicated text, no workspace
    del block
    torch.cuda.empty_cache()


def test_uneven_buckets_are_refused(E):
    """Two ranks over 'a' * (2^30 + 2^20): nearly every suffix falls in one bucket, so one slice would exceed the
    single-GPU limit -- ERANGE with the "too uneven" message."""
    from hkcsa import _lib, dist_sa
    n = (1 << 30) + (1 << 20)
    text = torch.full((n,), ord("a"), dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.HkcsaError) as e:
        dist_sa.emulate_distributed_suffix_array([text[: n // 2].clone(), text[n // 2:].clone()])
    assert e.value.code == _lib.ERANGE and "too uneven" in str(e.value)
    del text
    torch.cuda.empty_cache()
