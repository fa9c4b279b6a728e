"""The references of the succinct-primitive tests (tests/succinct_reference.py and device_reference.bits_rank /
bits_select) against the CPU oracle's restatement of the reference's SuccinctRankSelect and GolombRiceEncoder, and
against a block-by-block count, on small vectors.  Runs without a GPU."""
import math

import numpy as np
import pytest
import torch

import device_reference as R
import succinct_reference as S
from oracle import oracle as O

M_VALUES = (1, 2, 3, 7, 30)


def _run_lengths(m):
    """Runs of length m*j and m*j +- 1 for j = 0..3 (length 0 dropped)."""
    return sorted({v for j in range(4) for v in (m * j - 1, m * j, m * j + 1) if v > 0})


def _bitmaps():
    rng = np.random.RandomState(5)
    yield "empty", np.zeros(0, dtype=np.uint8)
    yield "one_zero", np.zeros(1, dtype=np.uint8)
    yield "one_one", np.ones(1, dtype=np.uint8)
    yield "all_zeros", np.zeros(1000, dtype=np.uint8)
    yield "all_ones", np.ones(1000, dtype=np.uint8)
    yield "random", (rng.random_sample(5000) < 0.5).astype(np.uint8)
    yield "sparse", (rng.random_sample(5000) < 0.02).astype(np.uint8)
    yield "bytes", rng.randint(0, 256, 3000).astype(np.uint8)          # any nonzero byte is a one
    runs = []                                          # run-heavy: long runs of ones between runs of zeros
    for _ in range(200):
        runs.append(np.zeros(rng.randint(1, 5), dtype=np.uint8))
        runs.append(np.ones(rng.geometric(0.02), dtype=np.uint8))
    yield "runs_closed_by_end", np.concatenate(runs)
    yield "runs_closed_by_zero", np.concatenate(runs + [np.zeros(1, dtype=np.uint8)])
    for m in M_VALUES:
        parts = []
        for v in _run_lengths(m):
            parts += [np.zeros(2, dtype=np.uint8), np.ones(v, dtype=np.uint8)]
        yield f"runs_of_m{m}", np.concatenate(parts)


BITMAPS = dict(_bitmaps())


@pytest.mark.parametrize("m", M_VALUES)
@pytest.mark.parametrize("name", sorted(BITMAPS))
def test_golomb_encode_matches_oracle(name, m):
    bits = BITMAPS[name]
    got, total = S.golomb_encode(torch.from_numpy(bits), m, chunk=64)    # a small chunk: runs cross chunk edges
    want = O.golomb_encode(bits, m)
    assert total == len(want) == got.numel()
    assert np.array_equal(got.numpy(), want)


@pytest.mark.parametrize("m", M_VALUES)
def test_golomb_encode_of_single_runs(m):
    """One run of each length m*j, m*j +- 1, alone and closed by the end of input."""
    for v in _run_lengths(m):
        for bits in (np.ones(v, dtype=np.uint8), np.concatenate([np.zeros(3, dtype=np.uint8), np.ones(v, np.uint8)])):
            got, total = S.golomb_encode(torch.from_numpy(bits), m, chunk=7)
            want = O.golomb_encode(bits, m)
            assert total == v // m + 1 + m == len(want)
            assert np.array_equal(got.numpy(), want), (m, v)


def test_ones_runs_across_chunks():
    rng = np.random.RandomState(3)
    bits = (rng.random_sample(4000) < 0.7).astype(np.uint8)
    s, v = S.ones_runs(torch.from_numpy(bits), chunk=33)
    rebuilt = np.zeros_like(bits)
    for a, k in zip(s.tolist(), v.tolist()):
        assert k > 0 and (a == 0 or bits[a - 1] == 0) and (a + k == len(bits) or bits[a + k] == 0)
        rebuilt[a:a + k] = 1
    assert np.array_equal(rebuilt, bits)


@pytest.mark.parametrize("name", sorted(BITMAPS))
def test_rank_and_select_match_oracle(name):
    """bits_rank at every position; bits_select for 1 <= k <= ones, and the conventions k = 0 -> 0, k > ones -> n."""
    bits01 = (BITMAPS[name] != 0).astype(np.uint8)
    n = len(bits01)
    rs = O.rank_support(bits01)
    t = torch.from_numpy(bits01)
    assert np.array_equal(R.bits_rank(t, torch.arange(n + 1), chunk=17).numpy(), rs.astype(np.int64))
    ones = int(rs[-1])
    ks = torch.arange(1, ones + 1)
    if ones:
        got = R.bits_select(t, ks, chunk=17).numpy()
        assert np.array_equal(got, [O.select(rs, int(k)) for k in ks])
    assert O.select(rs, 0) == 0
    assert O.select(rs, ones + 1) == n


def _brute_rrr(bits):
    n = len(bits)
    nblocks = -(-n // 15)
    ones = stream = 0
    for blk in range(nblocks):
        c = int(np.count_nonzero(bits[15 * blk:15 * blk + 15]))
        ones += c
        stream += math.ceil(math.log2(math.comb(15, c))) if math.comb(15, c) > 1 else 0
    return {"nbits": n, "nblocks": nblocks, "nsuper": -(-nblocks // 64), "ones": ones, "stream_bits": stream}


@pytest.mark.parametrize("n", [0, 1, 14, 15, 16, 959, 960, 961, 2000, 15 * 64 * 3 + 7])
@pytest.mark.parametrize("kind", ["random", "sparse", "ones", "bytes"])
def test_rrr_expected_matches_block_count(n, kind):
    rng = np.random.RandomState(n)
    bits = {"random": lambda: (rng.random_sample(n) < 0.5).astype(np.uint8),
            "sparse": lambda: (rng.random_sample(n) < 0.03).astype(np.uint8),
            "ones": lambda: np.ones(n, dtype=np.uint8),
            "bytes": lambda: rng.randint(0, 256, n).astype(np.uint8)}[kind]()
    assert S.rrr_expected(torch.from_numpy(bits), chunk=15 * 7) == _brute_rrr(bits)


def test_rrr_class_widths():
    assert S.rrr_class_widths().tolist() == [0, 4, 7, 9, 11, 12, 13, 13, 13, 13, 12, 11, 9, 7, 4, 0]


def test_all_patterns_vector_spells_every_block_once():
    v = S.all_patterns_vector().numpy().reshape(-1, 15)
    values = (v.astype(np.int64) << np.arange(15)).sum(1)
    assert np.array_equal(values, np.arange(1 << 15))
    exp = S.rrr_expected(torch.from_numpy(v.flatten()))
    assert exp["nsuper"] == 512 and exp["ones"] == 15 << 14
    assert exp["stream_bits"] == sum(math.comb(15, c) * S.rrr_class_widths()[c].item() for c in range(16))
