"""GPU parity of the drop-in Python API (csa/*.py, utils/*.py) against outputs frozen from the
reference itself (tests/golden/).  These read like the reference's own demos: same imports, same
calls, results compared with ==."""
import numpy as np
import pytest

from conftest import golden_case_names
from oracle import oracle as O

pytestmark = pytest.mark.gpu
CASES = golden_case_names()


@pytest.fixture(scope="module", autouse=True)
def _need_cuda(cuda):
    return cuda


def s(b: bytes) -> str:
    return b.decode("latin-1")


@pytest.mark.parametrize("name", CASES)
def test_suffix_array_bwt_count_occ(golden, name):
    from csa.suffix_array import build_suffix_array, ksa, optimized_ksa
    from csa.bwt import bwt_transform
    from utils.utils import build_count, build_occ
    text = s(golden.text(name))
    sa = build_suffix_array(text)
    assert isinstance(sa, list) and sa == golden.get(f"{name}/sa").tolist()
    assert ksa(text) == sa and optimized_ksa(text) == sa
    bwt = bwt_transform(text, sa)
    assert isinstance(bwt, str) and bwt == s(golden.get(f"{name}/bwt").tobytes())
    assert build_count(text) == {chr(int(k)): v for k, v in golden.meta[name]["count"].items()}
    keys = [k for k in golden.arr.files if k.startswith(f"{name}/occ/")]
    if keys:
        occ = build_occ(text)
        assert set(occ.keys()) == {chr(int(k.rsplit("/", 1)[1])) for k in keys}
        for k in keys:
            assert occ[chr(int(k.rsplit("/", 1)[1]))] == golden.get(k).tolist()


@pytest.mark.parametrize("name", CASES)
def test_wavelet_tree(golden, name):
    from csa.wavelet_tree import WaveletTree
    meta = golden.meta[name]
    if meta["n"] == 0:
        return
    text = s(golden.text(name))
    wt = WaveletTree(text)
    assert wt.text == text
    assert len(wt.tree) == len(wt.rank_structures) == meta["wt_levels"]
    assert wt.m == meta["wt_m"]
    assert [ord(c) for c in wt.alphabet] == meta["wt_alphabet_after"]
    for l, (compressed, left, right, next_text) in enumerate(wt.tree):
        assert [ord(c) for c in left] == meta["wt_left"][l]
        assert [ord(c) for c in right] == meta["wt_right"][l]
        assert len(next_text) == meta["wt_next_len"][l]
        assert "".join(next_text) == s(golden.get(f"{name}/wt/{l}/next").tobytes())
        rs = wt.rank_structures[l]
        n_l = int(golden.get(f"{name}/wt/{l}/nbits")[0])
        assert rs.n == n_l
        assert np.array_equal(rs.bit_vector, np.unpackbits(golden.get(f"{name}/wt/{l}/bits"))[:n_l])
        assert rs.bit_vector.dtype == np.uint8 and rs.rank_support.dtype == np.uint32
        if golden.has(f"{name}/wt/{l}/rank_support"):
            assert np.array_equal(rs.rank_support, golden.get(f"{name}/wt/{l}/rank_support"))
        for k, v in zip(golden.get(f"{name}/wt/{l}/select_k"), golden.get(f"{name}/wt/{l}/select_v")):
            assert rs.select(int(k)) == int(v)
        g_len = int(golden.get(f"{name}/wt/{l}/golomb_len")[0])
        want = np.unpackbits(golden.get(f"{name}/wt/{l}/golomb"))[:g_len].tolist()
        assert list(compressed) == want
    assert wt.compress() == [lvl[0] for lvl in wt.tree]
    assert wt.decompress(wt.compress()) == meta["wt_decompress"] == ""
    for i, v in meta["wt_rank_quirk"]:
        assert int(wt.rank("a", i)) == v                      # symbol ignored, last level answers
    for k, v in meta["wt_select_quirk"]:
        assert int(wt.select("a", k)) == v
    # correct symbol queries (extensions)
    arr = np.frombuffer(golden.text(name), dtype=np.uint8)
    for i in (0, len(arr) // 2, len(arr) - 1):
        assert wt.access(i) == text[i]
        assert wt.rank_c(text[i], i) == int((arr[:i] == arr[i]).sum())


def test_rank_select_and_golomb_classes(golden):
    from csa.wavelet_tree import SuccinctRankSelect, GolombRiceEncoder
    rs = SuccinctRankSelect([0, 1, 1, 0, 0, 1])
    assert [int(rs.rank(i)) for i in range(7)] == golden.meta["_rs_literal"]["rank"]
    assert [rs.select(k) for k in range(6)] == golden.meta["_rs_literal"]["select"]
    assert isinstance(rs.rank(3), np.uint32) and isinstance(rs.select(2), int)
    with pytest.raises(IndexError):
        rs.rank(7)
    for bitmap in ([1, 0, 1, 0, 1, 0], [0] * 9, [1] * 9, [1, 1, 0, 1, 1, 1, 0, 0, 1], [1] * 100 + [0] + [1] * 7):
        enc = GolombRiceEncoder(bitmap)
        b = np.asarray(bitmap, dtype=np.uint8)
        assert enc.m == O.golomb_m(int(b.sum()), len(b))
        assert enc.encode(bitmap) == O.golomb_encode(b, enc.m).tolist()
    assert GolombRiceEncoder([]).encode([]) == []


@pytest.mark.parametrize("name", CASES)
def test_enhanced_fm_index(golden, name):
    from csa.enhanced_fm_index import EnhancedFMIndex
    meta = golden.meta[name]
    if "fm_queries" not in meta:
        return
    text = s(golden.text(name))
    fm = EnhancedFMIndex(text)
    assert fm.text == text + "$"
    assert fm.suffix_array == golden.get(f"{name}/fm/sa").tolist()
    assert fm.bwt == s(golden.get(f"{name}/fm/bwt").tobytes())
    assert fm.count == {chr(int(k)): v for k, v in meta["fm_count"].items()}
    assert set(fm.occ.keys()) == set(fm.bwt)
    for q in meta["fm_queries"][:40]:
        p = s(bytes(q["p"]))
        assert fm.find_range(p) == (q["l"], q["r"])
        found = fm.find(p)
        assert len(found) == q["find_len"] and sum(found) == q["find_sorted_sum"]
        if q["find"] is not None:
            assert found == q["find"]
    qs = [s(bytes(q["p"])) for q in meta["fm_queries"]]
    lo, hi = fm.find_range_batch(qs)
    assert lo.tolist() == [q["l"] for q in meta["fm_queries"]] and hi.tolist() == [q["r"] for q in meta["fm_queries"]]
    assert fm.count_batch(qs).tolist() == [q["find_len"] for q in meta["fm_queries"]]
    for c, i, v in meta["fm_rank"]:
        assert fm.rank(chr(c), i) == v
    if len(fm.text) <= 3000:
        for ch in set(fm.bwt):
            assert fm.occ[ch] == O.occ_dense(fm.bwt.encode("latin-1"), ord(ch)).tolist()


@pytest.mark.parametrize("name", CASES)
def test_fmindex_and_compressed_suffix_array(golden, name):
    from csa.csa import FMIndex, CompressedSuffixArray
    meta = golden.meta[name]
    if "fmindex_rank_keys" not in meta:
        return
    text = s(golden.text(name))
    fi = FMIndex(text)
    assert fi.suffix_array == golden.get(f"{name}/sa").tolist()
    assert fi.bwt == s(golden.get(f"{name}/bwt").tobytes())
    assert [ord(k) for k in fi.rank.keys()] == meta["fmindex_rank_keys"]      # first-appearance order
    for k in fi.rank:
        key = f"{name}/fmindex/rank/{ord(k)}"
        if golden.has(key):
            assert fi.rank[k] == golden.get(key).tolist()
    assert len(fi.backward_search(text[:3])) == meta["fmindex_backward_search_len"]
    assert (fi.find_pattern(text[:3]) == fi.suffix_array) == meta["fmindex_find_pattern_is_sa"]
    if "fm_queries" in meta and "$" not in text:
        csa = CompressedSuffixArray(text, epsilon=0.5)
        assert csa.sa_sample_rate >= 1
        for q in meta["fm_queries"][:30]:
            p = s(bytes(q["p"]))
            got = csa.locate(p)
            assert got == sorted(got) and len(got) == q["find_len"] and sum(got) == q["find_sorted_sum"]
            assert csa.count(p) == q["find_len"]
            if q["find"] is not None:
                assert got == sorted(q["find"])


def test_reference_benchmark_workload():
    """tests/benchmark.py:110 default workload ("mississippi$" * 1000) through the API its benchmark
    expects; '$' inside the text, so compare with the oracle's EnhancedFMIndex restatement instead of
    brute force (SURVEY.md A.4)."""
    from csa.enhanced_fm_index import EnhancedFMIndex
    text = "mississippi$" * 1000
    fm = EnhancedFMIndex(text)
    t = text.encode() + b"$"
    sa = O.build_suffix_array(t)
    assert fm.suffix_array == sa.tolist()
    ofm = O.FM(O.bwt_transform(t, sa))
    for p in ("ssi", "mississippi$m", "i$", "$", "pp", "x", "", "mississippi$" * 3):
        l, r = ofm.find_range(p.encode())
        assert fm.find_range(p) == (l, r)
        assert fm.find(p) == ([] if l < 0 else sa[l:r + 1].tolist())


def test_error_behaviour_matches_reference():
    from csa.bwt import bwt_transform
    from csa.wavelet_tree import WaveletTree
    from csa.enhanced_fm_index import EnhancedFMIndex
    with pytest.raises(IndexError):
        bwt_transform("banana", [5, 3, 1])                    # suffix_array[i] past the end
    with pytest.raises(IndexError):
        bwt_transform("banana", [5, 3, 1, 0, 4, 9])           # text[pos] out of range
    assert bwt_transform("banana", [5, 3, 1, 0, 4, 2, 7, 7]) == "nnbaaa"   # extra entries ignored
    wt = WaveletTree("banana")
    with pytest.raises(IndexError):
        wt.rank("a", 6)                                       # rank_support[i + 1] past n
    with pytest.raises(IndexError):
        wt.run_length_encode([])
    assert WaveletTree("aaaa").rank("a", 2) == 0 and WaveletTree("aaaa").m is None
    fm = EnhancedFMIndex("banana")
    assert fm.find("nab") == [] and fm.find_range("x") == (-1, -1) and fm.find_range("") == (0, 6)
    assert fm.find("ana") == [3, 1] and fm.find_range("a$") == (1, 1)
    assert fm.rank("z", 3) == 0 and fm.rank("a", 100) == 3


def test_lazy_views_above_threshold(monkeypatch):
    """Force the large-n return types on a small input and check they still compare equal."""
    from hkcsa import views
    monkeypatch.setattr(views, "MATERIALIZE_MAX", 16)
    from csa.suffix_array import build_suffix_array
    from csa.bwt import bwt_transform
    from csa.enhanced_fm_index import EnhancedFMIndex
    from csa.wavelet_tree import WaveletTree
    text = O.gen_text(O.ENG96, 5, 3000).tobytes().decode("latin-1")
    sa = build_suffix_array(text)
    want = O.build_suffix_array(text)
    assert isinstance(sa, views.DeviceSequence) and sa == want.tolist() and sa[10] == int(want[10])
    assert bwt_transform(text, sa) == O.bwt_transform(text, want).tobytes().decode("latin-1")
    fm = EnhancedFMIndex(text)
    assert isinstance(fm.occ, views.OccView)
    ch = text[7]
    col = O.occ_dense(fm.bwt.encode("latin-1"), ord(ch))
    assert fm.occ[ch][100] == int(col[100]) and fm.occ[ch][90:95] == col[90:95].tolist() and len(fm.occ[ch]) == len(col)
    assert fm.occ[ch] == col.tolist()
    wt = WaveletTree(text)
    _, spine = O.wt_spine(text)
    assert isinstance(wt.tree[0][0], views.LazyList)
    assert list(wt.tree[0][0]) == O.golomb_encode(spine[0]).tolist()
    assert int(wt.rank_structures[0].rank(17)) == int(spine[0][:17].sum())


def _golden_hk():
    import json
    import os
    from conftest import ROOT
    with open(os.path.join(ROOT, "tests", "golden", "golden_hk.json")) as f:
        return json.load(f)


def test_high_order_entropy_matches_the_reference(golden):
    """H_k values frozen from the reference's own calculate_high_order_entropy (tests/golden/make_golden_hk.py imports
    it unmodified) for every golden text, k in {-1, 0, 1, 2, 3, 5, 8, 12, 20}: the GPU version (run heads on the
    suffix array, fp64 sums in a fixed order) must agree to 1e-9 relative -- only the summation order differs."""
    from csa.high_order_entropy import calculate_high_order_entropy, entropy_profile
    hk = _golden_hk()
    checked = 0
    for name, rec in hk.items():
        text = rec["text"] if "text" in rec else golden.text(name).decode("latin-1")
        for k_s, want in rec["hk"].items():
            got = calculate_high_order_entropy(text, int(k_s))
            assert got == pytest.approx(want, rel=1e-9, abs=1e-12), (name, k_s)
            checked += 1
        ks = [int(k) for k in rec["hk"] if int(k) >= 0]
        prof = entropy_profile(text, ks)                       # several orders from one suffix array
        for k in ks:
            assert prof[k] == pytest.approx(rec["hk"][str(k)], rel=1e-9, abs=1e-12), (name, k)
    assert checked >= 250
    assert calculate_high_order_entropy("", 2) == 0 and calculate_high_order_entropy("abc", -1) == 0
    assert calculate_high_order_entropy("abc", 5) == 0 and calculate_high_order_entropy("abc", 3) == 0


def test_high_order_entropy_is_bit_reproducible():
    from csa.high_order_entropy import calculate_high_order_entropy
    t = O.gen_text(O.ENG96, 3, 300_000).tobytes().decode("latin-1")
    assert len({calculate_high_order_entropy(t, 4) for _ in range(3)}) == 1


def test_text_beyond_latin1_is_recoded_order_preserving():
    """The reference compares Python strings (csa/suffix_array.py:132): code points above 255 are legal symbols.
    Here such a text is re-coded to bytes in code-point order; every result must equal the plain-Python definition."""
    from csa.suffix_array import build_suffix_array
    from csa.bwt import bwt_transform
    from csa.enhanced_fm_index import EnhancedFMIndex
    from utils.utils import build_count
    for text in ("αβγαβγδαβα" * 7 + "ω", "naïve café — 北京 naïve café — 北京 coöperate"):
        want_sa = sorted(range(len(text)), key=lambda i: text[i:])                 # csa/suffix_array.py:131-134
        sa = build_suffix_array(text)
        assert sa == want_sa
        want_bwt = "".join(text[i - 1] if i > 0 else text[-1] for i in want_sa)    # csa/bwt.py:3-13
        assert bwt_transform(text, sa) == want_bwt
        tot, want_count = 0, {}
        for c in sorted(set(text)):                                               # utils/utils.py:16-24
            want_count[c] = tot
            tot += text.count(c)
        assert build_count(text) == want_count
        fm = EnhancedFMIndex(text)
        t2 = text + "$"
        sa2 = sorted(range(len(t2)), key=lambda i: t2[i:])
        assert fm.text == t2 and fm.suffix_array == sa2
        assert fm.bwt == "".join(t2[i - 1] if i > 0 else t2[-1] for i in sa2)
        for q in (text[3:6], text[:2], "zz", "北", "\U0001F600", ""):
            occ = sorted(i for i in range(len(t2)) if t2.startswith(q, i)) if q else list(range(len(t2)))
            l, r = fm.find_range(q)
            assert (r - l + 1 if l >= 0 else 0) == len(occ), q
            assert sorted(fm.find(q)) == occ, q
        assert fm.rank(text[0], len(t2)) == t2.count(text[0]) and fm.rank("\U0001F600", 5) == 0


def test_patterns_with_unseen_code_points_are_misses():
    """csa/enhanced_fm_index.py:27-28: an unseen symbol makes the range (-1, -1); a pattern with a code point above
    255 on a latin-1 text is such a pattern (it used to raise)."""
    from csa.enhanced_fm_index import EnhancedFMIndex
    from csa.csa import CompressedSuffixArray
    fm = EnhancedFMIndex("banana bandana")
    assert fm.find_range("ba\u0107") == (-1, -1) and fm.find("\u4e2d") == []
    lo, hi = fm.find_range_batch(["ana", "\u0107", "ban"])
    assert lo.tolist()[1] == -1 and hi.tolist()[1] == -1 and lo.tolist()[0] >= 0 and lo.tolist()[2] >= 0
    csa = CompressedSuffixArray("banana bandana")
    assert csa.count("\u0107a") == 0 and csa.locate("\u0107a") == [] and csa.locate("ana") == [1, 3, 11]


def test_compressed_suffix_array_on_text_holding_the_sentinel(golden):
    """A text that already contains '$' has no unique sentinel: LF walks need not reach a sampled row (the LF walk is
    bounded and reports HKCSA_NO_POSITION instead of spinning).  CompressedSuffixArray then keeps the suffix array
    and answers what EnhancedFMIndex.find answers."""
    from csa.csa import CompressedSuffixArray
    from csa.enhanced_fm_index import EnhancedFMIndex
    for text in ("ab$ab", "mississippi$" * 40, golden.text("byte_16384").decode("latin-1")):
        csa = CompressedSuffixArray(text, sa_sample_rate=6)
        fm = EnhancedFMIndex(text)
        assert ("$" in text) == (not csa.sentinel_unique)
        for q in (text[:3], text[5:9], "$a", "$", "ssi"):
            assert csa.locate(q) == sorted(fm.find(q)), (text[:12], q)
            assert csa.count(q) == len(fm.find(q))


def test_lf_walk_is_bounded_when_the_sentinel_is_not_unique():
    """Sampled locate straight on the engine, on a text that holds its sentinel twice ('ab$ab' + '$', rate 6).  A plain
    LF step misranks the row of suffix 0 here (rows {2, 0, 4} would never reach the marked row 3); the kernels take
    the exact step, so every walk ends within `rate` steps at the position the suffix array holds."""
    import torch
    from hkcsa import engine as E
    d = E.to_device_u8(b"ab$ab$")
    idx = E.DeviceIndex(d, sa_sample_rate=6)
    rows = torch.arange(6, dtype=torch.int32, device=d.device)
    via_sa = idx.locate_rows(rows, use_samples=False).cpu().numpy().astype(np.uint32)
    assert via_sa.tolist() == sorted(range(6), key=lambda i: b"ab$ab$"[i:])
    for use_occ in (False, True):
        if use_occ:
            idx.build_occ_table(5, layout=1)
        got = idx.locate_rows(rows, use_samples=True).cpu().numpy().astype(np.uint32)
        assert got.tolist() == via_sa.tolist(), use_occ


def test_reference_benchmark_harness_runs_on_the_package(capsys):
    """SURVEY.md 8f row 1: the reference's tests/benchmark.py made runnable, as the package's restatement
    benchmarks/benchmark.py (utils.utils and csa.csa from this package).  run_full_benchmark on the reference's own
    default workload, "mississippi$" * 1000 (:110), must finish and locate what a plain scan finds."""
    from benchmarks import benchmark as bench
    text = "mississippi$" * 1000
    res = bench.run_full_benchmark(text, pattern_lengths=[5, 10, 50, 100, 500, 1000], iterations=2)
    bench.print_benchmark_summary(res)
    out = capsys.readouterr().out
    assert "Benchmark Summary" in out and sorted(res.pattern_times) == [5, 10, 50, 100, 500, 1000]
    assert res.construction_time > 0 and res.total_time >= res.construction_time
    # The benchmark text holds '$' itself, so the appended sentinel is not unique and backward search is the
    # reference's recurrence on a BWT whose rows are suffixes, not rotations (it reports e.g. one spurious row for
    # "mississippi$mi"): locate must return exactly what the reference-parity EnhancedFMIndex.find returns ...
    from csa.enhanced_fm_index import EnhancedFMIndex
    csa, _, _ = bench.benchmark_construction(text)
    fm = EnhancedFMIndex(text)
    for q in ("ssi", "mississippi$mi", text[7:507], "$m", "x"):
        locs, _, _ = bench.benchmark_pattern_search(csa, q)
        assert locs == sorted(fm.find(q)), q
    # ... and on the same text with a sentinel-free separator, what a plain scan finds
    clean = text.replace("$", "#")
    csa2, _, _ = bench.benchmark_construction(clean)
    for q in ("ssi", "mississippi#mi", clean[7:507], "#m", "x"):
        locs, _, _ = bench.benchmark_pattern_search(csa2, q)
        assert locs == [i for i in range(len(clean)) if clean.startswith(q, i)], q


def test_main_demo_matches_reference_output(capsys):
    """python main.py of the reference prints the whole suffix array for 'example' (its backward search is
    degenerate) and three Golomb lists of lengths 26 / 10 / 11 (SURVEY.md A.10)."""
    import importlib.util
    import os
    from conftest import PKG
    spec = importlib.util.spec_from_file_location("hk_main", os.path.join(PKG, "main.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.main()
    out = capsys.readouterr().out
    assert "Pattern 'example' found at indices: [7, 10, 4, 18, 13, 8, 17, 11, 20, 1, 5, 2, 16, 14, 9, 15, 6, 3, 22, 19, 0, 12, 21]" in out
    lists = eval(out.split("Wavelet Tree Compression: ")[1])
    assert [len(x) for x in lists] == [26, 10, 11]
