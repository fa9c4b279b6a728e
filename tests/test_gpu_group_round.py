"""The group round of the single-GPU suffix-array builder (round 1 without a radix sort) orders each small group of
round-0 survivors by comparing the text from the depth its members share.  A comparison that starts one symbol too
deep orders the members past the symbol that tells them apart; one that stops too early leaves them tied.

The texts plant families of repeats in random filler: a block, and 2..17 copies of it of which every other one carries
a single mutation at offset d = 0..48 from the block start.  The suffixes that start at the copies (and at every shift
inside them) form round-0 groups whose members first differ at d minus the shift, so some mutation lands in every
position of the key and
beyond it, in particular inside the gram or code word the key cuts.  Families sit at every offset of the
working set, hence across the 1008-element CTA stride of the group kernel, and one family ends the text.  Every build
asserts from its stats that the group round ran, and the suffix array and the BWT are checked against the oracle."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

FIN_MAX = 1024          # sa_finish_small_kernel takes at most this many suffixes
BLOCK = 72              # symbols of a planted block: longer than any key covers, plus the deepest mutation


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _alphabet(code: str) -> np.ndarray:
    if code == "gram":
        return np.frombuffer(b"ACGT", dtype=np.uint8)            # DNA + '$': the k-gram code (k = 6)
    return np.arange(30, 127, dtype=np.uint8)                    # 97 symbols: the per-symbol code


def _planted_text(code: str, n_filler: int, seed: int, sizes) -> bytes:
    alpha = _alphabet(code)
    rng = np.random.RandomState(seed)
    parts = []
    fams = [(d, c) for d in range(49) for c in sizes]
    rng.shuffle(fams)
    gap = n_filler // (len(fams) + 1)
    for i, (d, c) in enumerate(fams + [(int(rng.randint(0, 49)), int(sizes[-1]))]):
        block = rng.choice(alpha, BLOCK)
        for j in range(c):
            cp = block.copy()
            if j & 1:
                cp[d] = alpha[(np.searchsorted(alpha, cp[d]) + 1 + rng.randint(0, alpha.size - 1)) % alpha.size]
            parts.append(rng.choice(alpha, int(rng.randint(1, 8))))
            parts.append(cp)
        if i < len(fams):
            parts.append(rng.choice(alpha, gap))
    return np.concatenate(parts).tobytes() + b"$"            # the last family ends the text


def _check(E, text: bytes):
    d = E.to_device_u8(text)
    st = E.SaStats()
    sa = E.suffix_array(d, st).cpu().numpy().astype(np.uint32)
    st2 = E.SaStats()
    sa2, bwt = E.suffix_array_bwt(d, st2)
    # round 1 was the group round: no radix pass, more survivors than the single-CTA finish takes
    assert st.rounds >= 2 and st.round_passes[1] == 0 and st.round_elems[1] > FIN_MAX, \
        (int(st.rounds), [int(st.round_elems[i]) for i in range(int(st.rounds))])
    want = O.build_suffix_array(text)
    bad = np.flatnonzero(sa != want)
    assert bad.size == 0, f"{bad.size} wrong rows, first at {bad[:5]}"
    assert np.array_equal(sa2.cpu().numpy().astype(np.uint32), want), "suffix_array_bwt differs from the oracle"
    assert bwt.cpu().numpy().tobytes() == O.bwt_transform(text, want).tobytes(), "BWT differs from the oracle"
    return st


@pytest.mark.parametrize("seed", [1, 2])
def test_group_round_gram_code(E, seed):
    st = _check(E, _planted_text("gram", 600_000, seed, [2, 3, 4, 7, 16, 17]))
    assert st.gram_k > 0, "the text should be keyed by the k-gram code"


@pytest.mark.parametrize("seed", [1, 2])
def test_group_round_symbol_code(E, seed):
    st = _check(E, _planted_text("symbol", 600_000, seed, [2, 3, 5, 8, 16, 17]))
    assert st.gram_k == 0, "the text should be keyed by the per-symbol code"


def test_group_round_every_size(E):
    """Every group size 2..17 at every mutation offset."""
    _check(E, _planted_text("gram", 800_000, 3, list(range(2, 18))))
