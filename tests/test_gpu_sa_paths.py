"""Every path of the single-GPU suffix-array builder (hkcsa_sa_build / hkcsa_sa_bwt_build), each on a text built to
land on one of its thresholds, with the path asserted from the build's stats and the answer checked exactly.

The builder picks its route by hard thresholds: lazy ranks after round 0 (survivors * 4 <= n), the group round as
round 1 (survivors * 2 <= n, more than 1024 of them), groups of 2..16 ordered inside it (by their 16-symbol windows,
the serial form within 64 symbols, or left tied for the next round), the CTA that owns a group (1008-element stride),
the single-CTA finish once at most 1024 suffixes are left, lazy look-ups through the key samples in buckets of more
than 128 keys, the key ping-pong parity of the doubling rounds, the BWT carried in keys of at most 56 bits, and
aligned or unaligned text loads.  An off-by-one at any of them changes the suffix array only on texts that reach it,
so every case here asserts from hkcsa_sa_stats that it reached its path: a text that misses fails, it is not skipped.

The round-0 key is a data format that may change, so the texts are not derived from it.  They are calibrated: a
build reports the survivors of round 0 (round_elems[1]) and the shared depth k0, and the text is adjusted until it
hits its target.  Texts up to ~1 MB are checked against the CPU oracle, repetitive or larger ones against the exact
device references of tests/device_reference.py."""
import numpy as np
import pytest
import torch

import device_reference as R
from oracle import oracle as O

pytestmark = pytest.mark.gpu

FIN_MAX = 1024          # sa_finish_small_kernel takes at most this many suffixes
GS_DEPTH = 64           # symbols the serial form compares beyond the shared depth
CARRY_BITS0 = "56"      # round-0 keys of at most 56 bits carry the BWT symbol


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _dev(E, text: bytes) -> torch.Tensor:
    return E.to_device_u8(text)


# ------------------------------------------------------------------ builds, checks and path assertions
def _stats_tuple(st):
    r = int(st.rounds)
    return (r, [int(st.round_elems[i]) for i in range(r)], [int(st.round_passes[i]) for i in range(r)],
            int(st.lazy_ranks), int(st.k0), int(st.key_bits0), int(st.gram_k))


def _survivors(st) -> int:
    """Suffixes left after round 0 (0 when round 0 finished the job)."""
    return int(st.round_elems[1]) if st.rounds >= 2 else 0


def _check(E, text: bytes, d_text: torch.Tensor | None = None, carry: bool = True):
    """Both entry points on the text, checked exactly; returns (sa as numpy, stats of the BWT build).  The stats of the
    two builds must agree on the path: the BWT changes what is written, not how the suffixes are sorted."""
    d = d_text if d_text is not None else _dev(E, text)
    st = E.SaStats()
    sa = E.suffix_array(d, st)
    st2 = E.SaStats()
    sa2, bwt = E.suffix_array_bwt(d, st2)
    assert _stats_tuple(st) == _stats_tuple(st2)
    if carry:
        assert st2.bwt_carried == 1 and st2.key_bits0 <= 56, (st2.bwt_carried, st2.key_bits0)
    got = sa.cpu().numpy().astype(np.uint32)
    assert np.array_equal(got, sa2.cpu().numpy().astype(np.uint32)), "suffix_array and suffix_array_bwt differ"
    if len(text) <= (1 << 20):
        want = O.build_suffix_array(text)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"{bad.size} wrong rows, first at {bad[:5]}; stats {_stats_tuple(st)}"
        assert bwt.cpu().numpy().tobytes() == O.bwt_transform(text, want).tobytes(), "BWT differs from the oracle"
    else:
        R.check_suffix_array(d, sa)
        assert torch.equal(bwt, R.bwt_of(d, sa)), "BWT differs from text[SA - 1]"
    return got, st2


def _finish_round(st) -> int:
    """The round at which sa_finish_small_kernel took the remaining suffixes (it is always the last round)."""
    r = int(st.rounds) - 1
    assert r >= 1 and st.round_passes[r] == 0 and st.round_elems[r] <= FIN_MAX, _stats_tuple(st)
    return r


def _assert_group_round(st):
    """Round 1 was the group round (group_local_keys): no radix pass, more survivors than the finish takes."""
    assert st.rounds >= 3 and st.round_passes[1] == 0 and st.round_elems[1] > FIN_MAX, _stats_tuple(st)


def _assert_invariants(st):
    """Every build: the finish is the last round, and no round after round 0 but the group round and the finish
    skips the radix sort."""
    r_fin = _finish_round(st) if st.rounds >= 2 and st.round_elems[int(st.rounds) - 1] <= FIN_MAX else None
    for r in range(1, int(st.rounds)):
        if st.round_passes[r] == 0:
            assert r == r_fin or (r == 1 and st.round_elems[1] > FIN_MAX), _stats_tuple(st)


# ------------------------------------------------------------------ survivor counts by calibration
# Filler that leaves (almost) no round-0 survivors: uniform bytes over a large alphabet (per-symbol code) or over 16
# symbols (the k-gram code), and a run of a symbol the filler does not use.  The run symbol's count is fixed: the
# copies not in the run sit at isolated positions of the filler, so the byte histogram (and with it the per-symbol code
# and k0) stays put while the run grows, and the survivors move by one per step.
RUN_AT = 16
RUN_SLACK = 96          # run symbols beyond the target: a key covers at most 64 of them


def _alphabet(code: str):
    if code == "symbol":
        return np.arange(40, 140, dtype=np.uint8), 200      # 101 symbols: the per-symbol code
    return np.frombuffer(b"abcdefghijklmnop", dtype=np.uint8), ord("z")   # 17 symbols: the k-gram code


def _run_text(n: int, zc: int, L: int, seed: int, code: str) -> bytes:
    alpha, z = _alphabet(code)
    rng = np.random.RandomState(seed)
    t = rng.choice(alpha, n)
    q = _slots(n, zc)
    assert zc - L <= q.size, "text too short for the isolated run symbols"
    # run position RUN_AT + j and slot q[zc - 1 - j] hold the same filler symbol: whichever of the two the run symbol
    # takes, the other keeps it, so every byte's count is the same for all L
    j = np.arange(max(0, zc - q.size), zc)
    t[q[zc - 1 - j]] = t[RUN_AT + j]
    t[RUN_AT:RUN_AT + L] = z
    t[q[: zc - L]] = z
    return t.tobytes()


def _slots(n: int, zc: int) -> np.ndarray:
    """Isolated positions for the run symbols outside the run, behind the longest run."""
    return np.arange(RUN_AT + zc + 3, n, 4)


def _calibrate(E, target: int, make, lo: int, hi: int):
    """A run length L in [lo, hi] whose text leaves exactly `target` round-0 survivors: (text, stats of that build),
    or (None, the survivors seen per L) when no L does."""
    seen = {}
    L = target + 8
    for _ in range(60):
        L = min(max(L, lo), hi)
        if L in seen:
            break
        text = make(L)
        st = E.SaStats()
        E.suffix_array(_dev(E, text), st)
        got = _survivors(st)
        seen[L] = got
        if got == target:
            return text, st
        below = [x for x, g in seen.items() if g < target]
        above = [x for x, g in seen.items() if g > target]
        a = max(below) if below else lo - 1
        b = min(above) if above else hi + 1
        if b - a <= 1:
            break
        nxt = L + (target - got)
        L = nxt if a < nxt < b else (a + b) // 2
    return None, sorted(seen.items())


SURVIVOR_CASES = [
    # (target survivors, n): n >= 4 * target -> lazy ranks, n < 4 * target -> eager
    (2, 8192),
    (1023, 8192), (1024, 8192), (1025, 8192),
    (1023, 3000), (1024, 3000), (1025, 3000),
    (4096, 16384), (4097, 16384),               # n / 4 and n / 4 + 1
    (4096, 8192), (4097, 8192),                 # n / 2 and n / 2 + 1
]


@pytest.mark.parametrize("code", ["symbol", "gram"])
@pytest.mark.parametrize("target,n", SURVIVOR_CASES)
def test_survivors_after_round0_pick_the_path(E, target, n, code, monkeypatch):
    """Exactly `target` suffixes survive round 0, all in one group of more than 16 (the run): finish-small straight
    after round 0 (look-ups with first_round = 1 when lazy), the group round, or a radix round 1, with lazy or eager
    ranks -- each decided by its threshold and visible in the stats."""
    monkeypatch.setenv("HKCSA_BITS0", CARRY_BITS0)
    zc = target + RUN_SLACK
    tried = []
    for seed in range(100 + target, 103 + target):      # a code that changes with the run may step over the target
        text, seen = _calibrate(E, target, lambda L: _run_text(n, zc, L, seed, code),
                                max(1, zc - _slots(n, zc).size), zc)
        if text is not None:
            break
        tried.append(seen)
    else:
        pytest.fail(f"no run length leaves {target} survivors after round 0 (survivors per run length: {tried})")
    _, st = _check(E, text)
    assert _survivors(st) == target
    assert (st.gram_k >= 4) == (code == "gram"), st.gram_k
    lazy = target * 4 <= n
    assert st.lazy_ranks == (1 if lazy else 0), _stats_tuple(st)
    if target <= FIN_MAX:
        assert _finish_round(st) == 1 and st.rounds == 2
    elif target * 2 <= n:
        _assert_group_round(st)
        assert st.round_elems[2] <= target, _stats_tuple(st)
    else:
        assert st.round_passes[1] > 0 and st.round_elems[1] == target, _stats_tuple(st)
    _assert_invariants(st)


# ------------------------------------------------------------------ the group round
# c copies of a random string S, each followed by different filler: the suffixes at one offset of S form one group
# of c members.  With |S| = k0 + 64 + X, the groups at offsets o share |S| - o symbols: beyond the depth k0 that is
# under 16 (decided by the windows), 16..63 (the serial form decides), or 64 and more (tied: left to the doubling
# rounds).  Sizes that do not all divide 1008 put group starts at every phase of the CTA stride.
def _group_text(k0: int, sets, seed: int, alpha: np.ndarray, gap=(40, 260), first_at_start=False) -> bytes:
    """sets: (copies, extra) pairs, each a string S of k0 + 64 + extra symbols planted `copies` times.  One copy of
    the first set starts the text when first_at_start, one copy of the last set ends it."""
    rng = np.random.RandomState(seed)
    strings = [rng.choice(alpha, max(k0 + GS_DEPTH + extra, 4)).tobytes() for _, extra in sets]
    copies = [i for i, (c, _) in enumerate(sets) for _ in range(c)]
    rng.shuffle(copies)
    first = len(sets) - 1
    copies.remove(first)                  # one copy of the last set goes at the very end
    if first_at_start:
        copies.remove(0)
    parts = [strings[0]] if first_at_start else []
    for i in copies:
        parts.append(rng.choice(alpha, rng.randint(*gap)).tobytes())
        parts.append(strings[i])
    parts.append(rng.choice(alpha, rng.randint(*gap)).tobytes())
    parts.append(strings[first])
    return b"".join(parts)


def _k0(E, text: bytes) -> int:
    st = E.SaStats()
    E.suffix_array(_dev(E, text), st)
    return int(st.k0)


def _lcp(text: bytes, a: int, b: int) -> int:
    n, l = len(text), 0
    while a + l < n and b + l < n and text[a + l] == text[b + l]:
        l += 1
    return l


def _neighbour_lcp(text: bytes, sa: np.ndarray, isa: np.ndarray, i: int) -> int:
    r = int(isa[i])
    return max(_lcp(text, i, int(sa[r - 1])) if r > 0 else 0, _lcp(text, i, int(sa[r + 1])) if r + 1 < len(sa) else 0)


SIZES = (2, 3, 15, 16, 17, 18)
WIDE_ALPHA = np.arange(1, 256, dtype=np.uint8)


@pytest.mark.parametrize("after", ["radix", "finish"])
def test_group_round_mixed_group_sizes(E, after, monkeypatch):
    """Hundreds of groups of 2, 3, 15, 16, 17 and 18 over several 1008-element CTA strides, with groups decided by
    their windows, by the serial form, and tied beyond 64 symbols; one copy ends the text (windows reaching the end).
    After the group round more than 1024 survivors go on to a radix round, or at most 1024 to the finish (round 2)."""
    monkeypatch.setenv("HKCSA_BITS0", CARRY_BITS0)
    probe = _group_text(8, [(2, 8)], 1, WIDE_ALPHA)
    k0 = _k0(E, probe)
    if after == "radix":
        sets = [(c, 8) for c in SIZES for _ in range(2)]
    else:
        sets = [(c, 2) for c in (2, 3, 15, 16) for _ in range(2)] + [(17, -GS_DEPTH + 20)]
    text = _group_text(k0, sets, 7, WIDE_ALPHA)
    _, st = _check(E, text)
    assert st.k0 == k0
    _assert_group_round(st)
    m1 = int(st.round_elems[1])
    assert m1 >= 4 * 1008, f"only {m1} survivors: fewer than four CTA strides"
    if after == "radix":
        assert st.round_elems[2] > FIN_MAX and st.round_passes[2] > 0, _stats_tuple(st)
    else:
        assert _finish_round(st) == 2, _stats_tuple(st)
    # the group round decided groups (fewer survivors after it) but left the tied ones and those above 16
    assert 0 < st.round_elems[2] < m1, _stats_tuple(st)
    _assert_invariants(st)


def test_group_round_window_before_position_8(E, monkeypatch):
    """16-bit round-0 keys (k0 of one or two symbols) and a copy at the very start: a member's window starts before
    position 8, another one's runs past the end; both groups are ordered by the serial form."""
    monkeypatch.setenv("HKCSA_BITS0", "16")
    alpha = WIDE_ALPHA
    k0 = _k0(E, _group_text(2, [(2, 8)], 3, alpha, first_at_start=True))
    assert k0 < 8, k0
    text = _group_text(k0, [(2, 8), (3, 8), (5, 8), (16, 8), (9, 8), (4, 8)], 11, alpha, first_at_start=True,
                       gap=(150, 400))
    sa, st = _check(E, text)
    k0 = int(st.k0)
    assert st.key_bits0 == 16 and k0 < 8, _stats_tuple(st)
    _assert_group_round(st)
    _assert_invariants(st)
    isa = np.empty_like(sa)
    isa[sa] = np.arange(len(sa), dtype=sa.dtype)
    n = len(text)
    # a key of 16 bits covers at most 16 symbols: an SA neighbour sharing that many is in the same round-0 group
    starts = [i for i in range(0, 8 - k0) if _neighbour_lcp(text, sa, isa, i) >= st.key_bits0]
    assert starts, "no group member with its window before position 8"
    ends = [i for i in range(n - 24 - k0 + 1, n) if _neighbour_lcp(text, sa, isa, i) >= st.key_bits0]
    assert ends, "no group member with its window past the end"


# ------------------------------------------------------------------ lazy look-ups
def _runs_text(n: int, seed: int, code: str, runs: int = 40) -> bytes:
    """Filler without the run symbol, and `runs` runs of it (100..400 long, each followed by its own filler).  The
    suffixes that keep at least a key's worth of run symbols are one group of thousands; the run tails z^j x.. (every
    run, every j up to the key's reach) are singletons next to each other in suffix order, inside the buckets of the
    run symbol's prefixes, which hold thousands of keys for large j and a few for small j.  A doubling round looks up
    rank(i + h) for the group members i: tails at consecutive sorted positions, so some answers fall on a key sample
    (every 64th sorted key), some just after one, and an answer one off ties two members that differ."""
    alpha, z = _alphabet(code)
    rng = np.random.RandomState(seed)
    t = rng.choice(alpha, n)
    for p in rng.choice(n // 1024 - 1, runs, replace=False) * 1024:
        t[p:p + rng.randint(100, 400)] = z
    return t.tobytes()


@pytest.mark.parametrize("code", ["symbol", "gram"])
@pytest.mark.parametrize("n", [1 << 20, 3_000_017])
@pytest.mark.parametrize("group_round", [True, False])
def test_lazy_lookups_in_small_and_large_buckets(E, n, group_round, code, monkeypatch):
    """Lazy ranks and a later radix round: the look-ups of rank(i + h) search buckets of the sorted round-0 keys of
    every size, through the key samples above 128 keys.  Without the group round, round 1 is a radix round whose
    look-ups take the lower bound itself (first_round = 1)."""
    monkeypatch.setenv("HKCSA_BITS0", CARRY_BITS0)
    if not group_round:
        monkeypatch.setenv("HKCSA_NO_GROUP_ROUND", "1")
    text = _runs_text(n, 5 + n % 7, code)
    _, st = _check(E, text)
    assert (st.gram_k >= 4) == (code == "gram"), st.gram_k
    assert st.lazy_ranks == 1, _stats_tuple(st)
    assert _survivors(st) > FIN_MAX
    if group_round:
        _assert_group_round(st)
        assert st.round_passes[2] > 0, _stats_tuple(st)          # radix round 2 looks ranks up
    else:
        assert st.round_passes[1] > 0, _stats_tuple(st)          # radix round 1, first_round = 1
    _assert_invariants(st)


# ------------------------------------------------------------------ pass parity of the doubling rounds
def _periodic(n: int, period: int, seed: int) -> bytes:
    rng = np.random.RandomState(seed)
    unit = rng.randint(97, 123, period).astype(np.uint8).tobytes()
    return (unit * (n // period + 1))[:n]


def _repeated_block(n: int, seed: int) -> bytes:
    block = O.gen_text(O.ENG96, seed, 3000).tobytes()
    return (block * (n // len(block) + 1))[:n]


def _doubling_passes(n: int) -> int:
    return ((n - 1).bit_length() + n.bit_length() + 7) // 8       # key = (group start, rank + 1)


@pytest.mark.parametrize("n", [(1 << 16) - 1, 1 << 16, (1 << 20) - 1, 1 << 20])
@pytest.mark.parametrize("kind", ["periodic", "block"])
def test_doubling_rounds_pass_parity(E, n, kind, monkeypatch):
    """Long-LCP texts keep most suffixes through many doubling rounds; at n = 2^k - 1 and 2^k the key of a round
    takes one pass more, so the key ping-pong ends on either buffer."""
    monkeypatch.setenv("HKCSA_BITS0", CARRY_BITS0)
    text = _periodic(n, 13, n % 97) if kind == "periodic" else _repeated_block(n, 3)
    _, st = _check_large(E, _dev(E, text))
    passes = _doubling_passes(n)
    radix = [r for r in range(1, int(st.rounds)) if st.round_passes[r] > 0]
    assert len(radix) >= 2, _stats_tuple(st)
    assert all(st.round_passes[r] == passes for r in radix), (passes, _stats_tuple(st))
    assert st.round_passes[radix[0]] % 2 == passes % 2
    _assert_invariants(st)


def _check_large(E, d: torch.Tensor):
    """_check against the device references (periodic texts make the oracle's comparison sort quadratic)."""
    st = E.SaStats()
    sa = E.suffix_array(d, st)
    st2 = E.SaStats()
    sa2, bwt = E.suffix_array_bwt(d, st2)
    assert _stats_tuple(st) == _stats_tuple(st2)
    assert st2.bwt_carried == 1
    assert torch.equal(sa, sa2)
    R.check_suffix_array(d, sa)
    assert torch.equal(bwt, R.bwt_of(d, sa))
    return sa.cpu().numpy(), st2


# ------------------------------------------------------------------ unaligned text
def _views(E, text: bytes, offsets):
    """The text at the given storage offsets of one allocation (offset 0: 512-byte aligned)."""
    n = len(text)
    buf = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
    src = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda() if n else None
    for off in offsets:
        v = buf[off:off + n]
        v.copy_(src)
        assert v.data_ptr() % 16 == off % 16
        yield off, v


def _unaligned_matches_aligned(E, text: bytes, check_oracle: bool):
    d0 = _dev(E, text)
    st0 = E.SaStats()
    sa0, bwt0 = E.suffix_array_bwt(d0, st0)
    if check_oracle:
        want = O.build_suffix_array(text)
        assert np.array_equal(sa0.cpu().numpy().astype(np.uint32), want)
        assert bwt0.cpu().numpy().tobytes() == O.bwt_transform(text, want).tobytes()
    else:
        R.check_suffix_array(d0, sa0)
        assert torch.equal(bwt0, R.bwt_of(d0, sa0))
    for off, v in _views(E, text, range(1, 16)):
        st = E.SaStats()
        sa = E.suffix_array(v, st)
        assert torch.equal(sa, sa0), f"offset {off}: suffix array differs from the aligned build"
        sa2, bwt = E.suffix_array_bwt(v)
        assert torch.equal(sa2, sa0) and torch.equal(bwt, bwt0), f"offset {off}: BWT build differs"
        assert _stats_tuple(st) == _stats_tuple(st0), f"offset {off}: another path than the aligned build"
    return st0


@pytest.mark.parametrize("n", [2047, 2048, 2049, 3 * 2048 + 63, 3 * 2048 + 64, 3 * 2048 + 65])
@pytest.mark.parametrize("kind", [O.ENG96, O.DNA4])
def test_unaligned_text_views(E, kind, n):
    """A user's text[1:] reaches the builder as is: every pack tile takes the unaligned load path of its key source
    (per-symbol code for ENG96, k-gram code for DNA), and the sampled gram histogram its unaligned loads."""
    text = O.gen_text(kind, 17 + n % 11, n).tobytes()
    st = _unaligned_matches_aligned(E, text, True)
    assert (st.gram_k >= 4) == (kind == O.DNA4), st.gram_k


def test_unaligned_text_views_on_the_group_round_and_lazy_paths(E, monkeypatch):
    """The group-round and lazy look-up texts above, through the same views."""
    monkeypatch.setenv("HKCSA_BITS0", CARRY_BITS0)
    k0 = _k0(E, _group_text(8, [(2, 8)], 1, WIDE_ALPHA))
    text = _group_text(k0, [(c, 8) for c in SIZES], 7, WIDE_ALPHA)
    st = _unaligned_matches_aligned(E, text, True)
    _assert_group_round(st)
    st = _unaligned_matches_aligned(E, _runs_text(1 << 20, 9, "symbol"), False)
    assert st.lazy_ranks == 1 and st.round_passes[2] > 0, _stats_tuple(st)
