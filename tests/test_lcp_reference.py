"""The reference LCP array of the LCP tests (Kasai, tests/lcp_reference.py) against a direct comparison of adjacent
suffixes, on small random texts over alphabets of 1, 2, 4 and 256 symbols, with and without '$' (unique or repeated).
Runs without a GPU."""
import numpy as np
import pytest

from lcp_reference import lcp_kasai
from oracle import oracle as O


def _brute_lcp(t: bytes) -> np.ndarray:
    sa = sorted(range(len(t)), key=lambda i: t[i:])          # byte order, a proper prefix first
    out = np.zeros(len(t), dtype=np.uint32)
    for r in range(1, len(t)):
        a, b = t[sa[r - 1]:], t[sa[r]:]
        h = 0
        while h < min(len(a), len(b)) and a[h] == b[h]:
            h += 1
        out[r] = h
    return np.array(sa, dtype=np.uint32), out


def _texts():
    rng = np.random.RandomState(11)
    for sigma in (1, 2, 4, 256):
        alpha = np.arange(97, 97 + sigma, dtype=np.uint8) if sigma < 256 else np.arange(256, dtype=np.uint8)
        for k in range(60):
            n = int(rng.randint(0, 200))
            body = alpha[rng.randint(0, sigma, size=n)].tobytes()
            for form in ("plain", "sentinel", "dollars"):
                if form == "plain":
                    yield f"s{sigma}_{k}_{form}", body
                elif form == "sentinel":
                    yield f"s{sigma}_{k}_{form}", body + b"$"
                elif k % 3 == 0:
                    cut = n // 2
                    yield f"s{sigma}_{k}_{form}", body[:cut] + b"$" + body[cut:] + b"$"


TEXTS = dict(_texts())
TEXTS.update({"mississippi_x40": b"mississippi$" * 40 + b"$", "ab$ab$": b"ab$ab$", "empty": b"", "one": b"$"})


@pytest.mark.parametrize("name", sorted(TEXTS))
def test_kasai_matches_direct_comparison(name):
    t = TEXTS[name]
    sa, want = _brute_lcp(t)
    assert np.array_equal(O.build_suffix_array(t), sa)
    assert np.array_equal(lcp_kasai(t, sa), want)


def test_kasai_refuses_a_suffix_array_of_the_wrong_length():
    with pytest.raises(ValueError):
        lcp_kasai(b"abc$", np.array([3, 0], dtype=np.uint32))
