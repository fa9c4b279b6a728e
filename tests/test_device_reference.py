"""CPU: the plain torch references of tests/device_reference.py agree with the oracle and the frozen reference outputs,
and each one rejects a corrupted answer -- what makes the GPU tests that use them (tests/test_gpu_envelope.py) fail on a
subtly wrong kernel.  Also the single-GPU size limit of every C entry point that plans a structure for n symbols."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import device_reference as R
from conftest import ROOT, golden_case_names
from oracle import oracle as O


def _t(b) -> torch.Tensor:
    return torch.from_numpy(np.frombuffer(bytes(b), dtype=np.uint8).copy())


def _fib(n):
    a, b = "a", "ab"
    while len(b) < n:
        a, b = b, b + a
    return b[:n].encode()


def _all_bytes(n, seed=6):
    alpha = np.array([b for b in range(256) if b != 0x24], dtype=np.uint8)
    body = alpha[np.random.RandomState(seed).randint(0, alpha.size, size=n)]
    body[: alpha.size] = alpha                      # every one of the 255 symbols occurs
    return body.tobytes()


TEXTS = {
    "banana": lambda: b"banana$",
    "sigma1": lambda: b"$",
    "all_a": lambda: b"a" * 3000 + b"$",
    "dna": lambda: O.gen_text(O.DNA4, 3, 20_000).tobytes() + b"$",
    "eng": lambda: O.gen_text(O.ENG96, 4, 20_000).tobytes() + b"$",
    "bytes255": lambda: _all_bytes(20_000) + b"$",
    "periodic": lambda: b"abcab" * 999 + b"$",
    "fibonacci": lambda: _fib(10_000) + b"$",
    "mississippi_inner": lambda: b"mississippi$" * 400 + b"$",
    "period11": lambda: (b"mississippi" * 400)[:4000] + b"$",
    "sentinel_not_minimal": lambda: b"\x01\x00\x02\x01\x00" * 300 + b"$",
}


def _sa(text: bytes) -> torch.Tensor:
    return torch.from_numpy(O.build_suffix_array(text).astype(np.int32))


# ------------------------------------------------------------------ agreement
@pytest.mark.parametrize("name", golden_case_names())
def test_checker_accepts_golden_suffix_arrays(golden, name):
    text = golden.text(name)
    sa = torch.from_numpy(golden.get(f"{name}/sa").astype(np.int32))
    isa = R.check_suffix_array(_t(text), sa)
    if len(text):
        assert np.array_equal(isa.numpy()[sa.numpy()], np.arange(len(text)))
        assert R.bwt_of(_t(text), sa).numpy().tobytes() == golden.get(f"{name}/bwt").tobytes()


@pytest.mark.parametrize("name", list(TEXTS))
def test_references_agree_with_the_oracle(name):
    text = TEXTS[name]()
    n = len(text)
    t, sa = _t(text), _sa(text)
    isa = R.check_suffix_array(t, sa, chunk=777)                 # chunk edges inside the text
    bwt = R.bwt_of(t, sa, chunk=1000)
    want_bwt = O.bwt_transform(text, sa.numpy().astype(np.uint32))
    assert np.array_equal(bwt.numpy(), want_bwt)
    # occ against the oracle's FM rank, at every position for two symbols and at random (symbol, position) pairs
    groups = R.symbol_positions(bwt, chunk=999)
    fm = O.FM(want_bwt)
    present = np.flatnonzero(np.bincount(want_bwt, minlength=256))
    rng = np.random.RandomState(1)
    sym = np.concatenate([np.repeat(present[:2], n + 1), rng.choice(present, 3000)]).astype(np.uint8)
    pos = np.concatenate([np.tile(np.arange(n + 1), min(2, len(present))), rng.randint(0, n + 1, 3000)])
    got = R.occ_at(bwt, torch.from_numpy(sym), torch.from_numpy(pos), groups).numpy()
    for c in present[:2]:
        dense = O.occ_dense(want_bwt, int(c)).astype(np.int64)
        assert np.array_equal(got[sym == c][: n + 1], dense)
    assert all(got[q] == fm.rank(int(sym[q]), int(pos[q])) for q in range(len(sym) - 3000, len(sym)))
    # LF^-1 grouping is the oracle's position lists
    opos, ostart = O.symbol_positions(want_bwt)
    assert np.array_equal(groups[0].numpy(), opos.astype(np.int32)) and np.array_equal(groups[1].numpy(), ostart)
    # pattern ranges: substrings, mutated substrings, absent symbols, the empty pattern, suffixes of the text
    pats, off = O.gen_patterns(5, 400, np.frombuffer(text[:-1] or b"a", dtype=np.uint8), 1, 64)
    extra = [b"", text[-3:], text[-1:], text[-64:], b"\xfe\xfd", text[:5]]
    flat = np.concatenate([pats, np.frombuffer(b"".join(extra), dtype=np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([len(e) for e in extra])]).astype(np.int64)
    # find_range counts cyclic occurrences and, past a non-final sentinel, follows LF: keep the patterns for which
    # suffix ranges and backward search are the same question (the sentinel at most as the last symbol)
    keep = [q for q in range(len(off) - 1) if b"$" not in flat[off[q]:off[q + 1] - 1].tobytes()]
    flat = np.concatenate([flat[off[q]:off[q + 1]] for q in keep] + [np.zeros(0, np.uint8)])
    off = np.concatenate([[0], np.cumsum([off[q + 1] - off[q] for q in keep])]).astype(np.int64)
    lo, hi = R.sa_range(t, sa, torch.from_numpy(flat), torch.from_numpy(off))
    w_lo, w_hi = fm.find_range_batch(flat, off)
    assert np.array_equal(lo.numpy(), w_lo) and np.array_equal(hi.numpy(), w_hi)
    # bit-vector rank / select against the oracle's restatement of the reference (every position, every one)
    for bits in O.wt_spine(want_bwt)[1][:2]:
        rs = O.rank_support(bits).astype(np.int64)
        b = torch.from_numpy(bits)
        assert np.array_equal(R.bits_rank(b, torch.arange(len(bits) + 1), chunk=333).numpy(), rs)
        ks = np.arange(1, int(rs[-1]) + 1)
        assert np.array_equal(R.bits_select(b, torch.from_numpy(ks), chunk=333).numpy(),
                              np.searchsorted(rs, ks, side="left"))
    # the invertibility criterion agrees with a direct LF inversion of the text
    inv = np.empty(n, dtype=np.int64)
    lf = np.empty(n, dtype=np.int64)
    lf[groups[0].numpy()] = np.arange(n)
    j = int(isa[0])
    for k in range(n - 1, -1, -1):
        inv[k] = want_bwt[j]
        j = lf[j]
    assert R.lf_invertible(bwt, isa) == (inv.astype(np.uint8).tobytes() == text)


# ------------------------------------------------------------------ the int64 forms (texts past 2^31 - 1 symbols)
def test_row_dtype_switches_past_int32():
    assert R._row_dtype(R.INT32_MAX, None) == torch.int32 and R._row_dtype(R.INT32_MAX + 1, None) == torch.int64
    assert R._row_dtype(5, True) == torch.int64 and R._row_dtype(5, False) == torch.int32


@pytest.mark.parametrize("name", golden_case_names())
def test_int64_checker_accepts_golden_suffix_arrays(golden, name):
    text = golden.text(name)
    sa = torch.from_numpy(golden.get(f"{name}/sa").astype(np.int64))
    isa = R.check_suffix_array(_t(text), sa, wide=True)
    assert isa.dtype == torch.int64
    if len(text):
        assert np.array_equal(isa.numpy()[sa.numpy()], np.arange(len(text)))
        assert R.bwt_of(_t(text), sa).numpy().tobytes() == golden.get(f"{name}/bwt").tobytes()


@pytest.mark.parametrize("name", list(TEXTS))
def test_int64_references_agree_with_the_oracle(name):
    """An int64 suffix array through every reference, with the int64 ISA and row lists forced: the same answers as the
    int32 forms and the oracle."""
    text = TEXTS[name]()
    n = len(text)
    t, sa32 = _t(text), _sa(text)
    sa = sa32.long()
    isa = R.check_suffix_array(t, sa, chunk=777, wide=True)
    assert isa.dtype == torch.int64 and torch.equal(isa, R.check_suffix_array(t, sa32).long())
    bwt = R.bwt_of(t, sa, chunk=1000)
    want_bwt = O.bwt_transform(text, sa32.numpy().astype(np.uint32))
    assert np.array_equal(bwt.numpy(), want_bwt)
    groups = R.symbol_positions(bwt, chunk=999, wide=True)
    opos, ostart = O.symbol_positions(want_bwt)
    assert groups[0].dtype == torch.int64
    assert np.array_equal(groups[0].numpy(), opos.astype(np.int64)) and np.array_equal(groups[1].numpy(), ostart)
    present = np.flatnonzero(np.bincount(want_bwt, minlength=256))
    rng = np.random.RandomState(2)
    sym = rng.choice(present, 3000).astype(np.uint8)
    pos = rng.randint(0, n + 1, 3000)
    got = R.occ_at(bwt, torch.from_numpy(sym), torch.from_numpy(pos), groups).numpy()
    fm = O.FM(want_bwt)
    assert all(got[q] == fm.rank(int(sym[q]), int(pos[q])) for q in range(3000))
    pats, off = O.gen_patterns(6, 300, np.frombuffer(text[:-1] or b"a", dtype=np.uint8), 1, 64)
    lo, hi = R.sa_range(t, sa, torch.from_numpy(pats), torch.from_numpy(off))
    lo32, hi32 = R.sa_range(t, sa32, torch.from_numpy(pats), torch.from_numpy(off))
    assert torch.equal(lo, lo32) and torch.equal(hi, hi32)
    keep = [q for q in range(len(off) - 1) if b"$" not in pats[off[q]:off[q + 1] - 1].tobytes()]
    w_lo, w_hi = fm.find_range_batch(pats, off)
    assert np.array_equal(lo.numpy()[keep], w_lo[keep]) and np.array_equal(hi.numpy()[keep], w_hi[keep])
    assert R.lf_invertible(bwt, isa) == R.lf_invertible(bwt, isa.int())


def test_int64_references_see_a_flipped_row():
    """The int64 row lists and occ reject what the int32 ones reject: a row moved to another symbol's list."""
    text = MUT_TEXT
    t, sa = _t(text), _sa(text).long()
    bwt = R.bwt_of(t, sa)
    pos, start = R.symbol_positions(bwt, wide=True)
    bad = bwt.clone()
    bad[1234] = bwt[1235] if bwt[1235] != bwt[1234] else bwt[0]
    assert not torch.equal(R.symbol_positions(bad, wide=True)[0], pos)
    q = torch.arange(len(text) + 1)
    c = torch.full_like(q, int(bwt[1234])).to(torch.uint8)
    assert not torch.equal(R.occ_at(bad, c, q), R.occ_at(bwt, c, q, (pos, start)))


def _golden_hk_cases():
    with open(os.path.join(ROOT, "tests", "golden", "golden_hk.json")) as f:
        d = json.load(f)
    out = []
    for name, v in sorted(d.items()):
        if "text" in v:
            try:
                text = v["text"].encode("latin-1")
            except UnicodeEncodeError:
                continue                                          # code points above 255: not a byte text
        else:
            text = None
        out.append((name, text, v["hk"]))
    return out


@pytest.mark.parametrize("name,text,hk", _golden_hk_cases(), ids=[c[0] for c in _golden_hk_cases()])
def test_entropy_matches_the_reference(golden, name, text, hk):
    text = golden.text(name) if text is None else text
    t = _t(text)
    sigma = len(set(text))
    for k, want in hk.items():
        k = int(k)
        if k > 7 and (k + 1) * max(1, (sigma - 1).bit_length()) > 64:
            continue                                              # does not pack into 64 bits
        got = R.entropy_hk(t, k, chunk=500)
        assert got == pytest.approx(want, rel=1e-9, abs=1e-12), (name, k)


def test_entropy_packs_twenty_symbol_contexts_on_dna():
    text = O.gen_text(O.DNA4, 7, 30_000).tobytes() + b"$"
    for k in (8, 12, 20):
        w = [text[i:i + k + 1] for i in range(len(text) - k)]
        from collections import Counter
        g, c = Counter(w), Counter(x[:k] for x in w)
        want = (sum(v * np.log2(v) for v in c.values()) - sum(v * np.log2(v) for v in g.values())) / len(text)
        assert R.entropy_hk(_t(text), k) == pytest.approx(want, rel=1e-12)


@pytest.mark.parametrize("text,want", [(b"a$b$", True), (b"ab$ab$", False), (b"mississippi$" * 40 + b"$", False),
                                       (b"banana$", True)])
def test_lf_invertible_matches_design(text, want):
    t, sa = _t(text), _sa(text)
    isa = R.check_suffix_array(t, sa)
    assert R.lf_invertible(R.bwt_of(t, sa), isa) is want


@pytest.mark.parametrize("name", list(TEXTS))
def test_exact_lf_step_of_locate(name):
    """The LF step the locate kernels take (csrc/common.cuh lf_fix): C[c] + occ(c, j), except that with j0 = ISA[0]
    and c0 = bwt[j0], row j0 steps to C[c0] and every c0-row before j0 to C[c0] + occ + 1.  It must equal
    ISA[SA[j] - 1 mod n] on every text, including those that hold their last symbol elsewhere."""
    text = TEXTS[name]()
    n = len(text)
    t, sa = _t(text), _sa(text)
    isa = R.check_suffix_array(t, sa)
    bwt = R.bwt_of(t, sa)
    groups = R.symbol_positions(bwt)
    rows = torch.arange(n)
    start = groups[1]
    plain = start[bwt.long()] + R.occ_at(bwt, bwt, rows, groups)
    j0 = int(isa[0])
    c0 = int(bwt[j0])
    fix = R.occ_at(bwt, bwt[j0:j0 + 1], torch.tensor([j0]), groups).item() != 0
    exact = plain.clone()
    if fix:
        before = (bwt == c0) & (rows < j0)
        exact[before] += 1
        exact[j0] = start[c0]
    want = isa[(sa.long() - 1) % n].long()
    assert torch.equal(exact, want)
    assert fix == (not R.lf_invertible(bwt, isa))
    assert torch.equal(plain, want) == (not fix)          # the plain step is wrong exactly when the fix applies


# ------------------------------------------------------------------ mutations: each reference rejects a wrong answer
MUT_TEXT = O.gen_text(O.ENG96, 12, 5000).tobytes() + b"$"


def _reject(text: bytes, sa: np.ndarray, match: str):
    """Both forms of the checker: an int32 suffix array with the int32 ISA, and an int64 one with the int64 ISA that
    texts past 2^31 - 1 symbols take."""
    with pytest.raises(AssertionError, match=match):
        R.check_suffix_array(_t(text), torch.from_numpy(sa.astype(np.int32)), chunk=701)
    with pytest.raises(AssertionError, match=match):
        R.check_suffix_array(_t(text), torch.from_numpy(sa.astype(np.int64)), chunk=701, wide=True)


def test_checker_rejects_two_adjacent_rows_with_equal_first_symbol_swapped():
    sa = O.build_suffix_array(MUT_TEXT).astype(np.int64)
    first = np.frombuffer(MUT_TEXT, dtype=np.uint8)[sa]
    i = int(np.flatnonzero(first[:-1] == first[1:])[1234])
    sa[[i, i + 1]] = sa[[i + 1, i]]
    _reject(MUT_TEXT, sa, f"out of order at row {i}")


def test_checker_rejects_rows_swapped_far_apart():
    sa = O.build_suffix_array(MUT_TEXT).astype(np.int64)
    sa[[10, 4000]] = sa[[4000, 10]]
    _reject(MUT_TEXT, sa, "out of order at row 10")


def test_checker_rejects_a_duplicated_entry():
    sa = O.build_suffix_array(MUT_TEXT).astype(np.int64)
    sa[2500] = sa[2501]
    _reject(MUT_TEXT, sa, "not a permutation")
    sa = O.build_suffix_array(MUT_TEXT).astype(np.int64)
    sa[77] = len(MUT_TEXT)
    _reject(MUT_TEXT, sa, "out of")


def test_checker_rejects_a_rotated_suffix_array():
    sa = O.build_suffix_array(MUT_TEXT).astype(np.int64)
    _reject(MUT_TEXT, np.roll(sa, 1), "out of order")
    _reject(MUT_TEXT, (sa + 1) % len(MUT_TEXT), "out of order")


def test_checker_rejects_the_wrong_tie_break_with_the_sentinel_inside():
    """'$' inside the text: the suffixes '$' (last) and '$$'/'$m...' share their first symbol.  Sorting the text as
    if it were cyclic, or a proper prefix last, are both wrong and both caught."""
    for text in (b"ab$ab$", b"mississippi$" * 40 + b"$", b"a$a$a$"):
        sa = O.build_suffix_array(text).astype(np.int64)
        n = len(text)
        rot = sorted(range(n), key=lambda i: text[i:] + text[:i])            # rotation order
        if rot != sa.tolist():
            _reject(text, np.array(rot), "out of order")
        longer_first = sorted(range(n), key=lambda i: text[i:] + b"\xff" * (n - (n - i)))
        if longer_first != sa.tolist():
            _reject(text, np.array(longer_first), "out of order")
        assert rot != sa.tolist() or longer_first != sa.tolist()


def test_range_and_bwt_comparisons_catch_off_by_one_and_flipped_bytes():
    """The GPU tests compare ranges and BWT bytes with torch.equal: an off-by-one range or one flipped BWT byte is a
    difference they see."""
    text = MUT_TEXT
    t, sa = _t(text), _sa(text)
    bwt = R.bwt_of(t, sa)
    bad = bwt.clone()
    bad[1234] ^= 1
    assert not torch.equal(bad, bwt)
    pats, off = O.gen_patterns(3, 300, np.frombuffer(text[:-1], dtype=np.uint8), 2, 12)
    lo, hi = R.sa_range(t, sa, torch.from_numpy(pats), torch.from_numpy(off))
    w_lo, w_hi = O.FM(bwt.numpy()).find_range_batch(pats, off)
    assert np.array_equal(lo.numpy(), w_lo) and np.array_equal(hi.numpy(), w_hi)
    hit = int(np.flatnonzero(w_lo >= 0)[0])
    for dlo, dhi in ((1, 0), (0, 1), (-1, 0), (0, -1)):
        a, b = w_lo.copy(), w_hi.copy()
        a[hit] += dlo
        b[hit] += dhi
        assert not (np.array_equal(lo.numpy(), a) and np.array_equal(hi.numpy(), b))


def test_entropy_and_invertibility_see_a_one_symbol_change():
    text = bytearray(O.gen_text(O.DNA4, 2, 4000).tobytes() + b"$")
    h = R.entropy_hk(_t(bytes(text)), 3)
    text[1000] = ord("A") if text[1000] != ord("A") else ord("C")
    assert R.entropy_hk(_t(bytes(text)), 3) != pytest.approx(h, rel=1e-9)
    t = _t(b"a$b$")
    sa = _sa(b"a$b$")
    isa = R.check_suffix_array(t, sa)
    bwt = R.bwt_of(t, sa)
    bwt2 = bwt.clone()
    j0 = int(isa[0])
    bwt2[0] = bwt[j0]                                          # a copy of bwt[j0] ahead of row j0
    assert j0 > 0 and R.lf_invertible(bwt, isa) and not R.lf_invertible(bwt2, isa)


# ------------------------------------------------------------------ the limit of the C entry points (no GPU)
def test_every_planning_entry_point_refuses_n_beyond_the_single_gpu_limit():
    from hkcsa import _lib
    L = _lib.load()
    big = _lib.MAX_N + 1
    hist = np.zeros(256, dtype=np.uint64)
    hist[ord("a")], hist[ord("$")] = big - 1, 1
    wt = _lib.WtPlan()
    assert L.hkcsa_wt_plan_from_hist(hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(wt)) == _lib.ERANGE
    hist[ord("a")] -= 1
    assert L.hkcsa_wt_plan_from_hist(hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(wt)) == _lib.OK
    assert wt.n == _lib.MAX_N
    assert L.hkcsa_bitvec_plan(big, C.byref(wt)) == _lib.ERANGE
    assert L.hkcsa_bitvec_plan(_lib.MAX_N, C.byref(wt)) == _lib.OK
    ssa = _lib.SsaPlan()
    assert L.hkcsa_ssa_plan_make(big, 32, C.byref(ssa)) == _lib.ERANGE
    assert L.hkcsa_ssa_plan_make(_lib.MAX_N, 1, C.byref(ssa)) == _lib.OK and ssa.n_samples == _lib.MAX_N
    occ = _lib.OccPlan()
    for layout in (0, 1):
        assert L.hkcsa_occ_plan_make(big, 97, 5, layout, C.byref(occ)) == _lib.ERANGE
        assert L.hkcsa_occ_plan_make(_lib.MAX_N, 97, 5, layout, C.byref(occ)) == _lib.OK
    # the builders refuse before touching a pointer (none of these is a device address)
    fake = C.c_void_p(0x1000)
    st = _lib.SaStats()
    assert L.hkcsa_sa_build(fake, big, fake, fake, 1 << 40, None, C.byref(st)) == _lib.ERANGE
    assert L.hkcsa_sa_bwt_build(fake, big, fake, fake, fake, 1 << 40, None, C.byref(st)) == _lib.ERANGE
    assert b"HKCSA_MAX_N" in L.hkcsa_last_error()


def test_engine_refuses_a_text_beyond_the_limit_before_any_kernel(monkeypatch):
    """DeviceIndex, suffix_array and suffix_array_bwt check n first; a meta tensor has a length and no storage, so a
    kernel launch or an allocation of its size would fail differently."""
    from hkcsa import _lib, engine
    big = torch.empty(_lib.MAX_N + 1, dtype=torch.uint8, device="meta")
    monkeypatch.setattr(engine, "_require_cuda", lambda: torch.device("meta"))
    for fn in (engine.DeviceIndex, engine.suffix_array, engine.suffix_array_bwt):
        with pytest.raises(_lib.HkcsaError) as e:
            fn(big)
        assert e.value.code == _lib.ERANGE
