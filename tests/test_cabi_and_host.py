"""CPU-only: the C-ABI library loads and exports every symbol include/hkcsa.h declares (no compute
calls), struct mirrors match, host-side planning logic, the lazy views, and the drop-in modules'
API surface."""
import ctypes as C
import inspect
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import oracle as O


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "hkcsa.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hkcsa_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from hkcsa import _lib
    L = _lib.load()
    names = _declared_functions()
    assert len(names) >= 35
    for name in names:
        assert hasattr(L, name), f"libhkcsa.so does not export {name}"
        assert name in _lib.SIGNATURES, f"ctypes binding lacks {name}"
    assert sorted(_lib.SIGNATURES) == names
    assert L.hkcsa_abi_version() == 1


def test_struct_mirrors_match_c_layout():
    from hkcsa import _lib
    L = _lib.load()
    for idx, st in enumerate((_lib.SaStats, _lib.WtPlan, _lib.SsaPlan, _lib.ProfEntry, _lib.OccPlan, _lib.DsaPlan,
                              _lib.RrrPlan)):
        assert L.hkcsa_struct_size(idx) == C.sizeof(st)


def test_scratch_queries_are_host_only():
    from hkcsa import _lib
    L = _lib.load()
    n = 1_000_000
    assert L.hkcsa_sa_scratch_bytes(n) >= 40 * n
    assert L.hkcsa_sa_scratch_bytes(2 * n) > L.hkcsa_sa_scratch_bytes(n)
    assert L.hkcsa_sort_scratch_bytes(n) > 0
    assert L.hkcsa_golomb_scratch_bytes(n) > 0


def _plan(seq: bytes):
    from hkcsa import _lib
    L = _lib.load()
    hist = np.bincount(np.frombuffer(seq, dtype=np.uint8), minlength=256).astype(np.uint64)
    p = _lib.WtPlan()
    assert L.hkcsa_wt_plan_from_hist(hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(p)) == 0
    return p


@pytest.mark.parametrize("seq", [b"banana", b"abcde", b"abcd", b"this is an example text", b"a", b"",
                                 bytes(range(256)) * 2, bytes(range(97)) * 3])
def test_wavelet_plan_matches_reference_split_rule(seq):
    """Tree shape (host logic of K3): the left-most node of every level must be the reference's
    alphabet halving (csa/wavelet_tree.py:78-80), checked against the oracle's spine."""
    p = _plan(seq)
    alpha, spine = O.wt_spine(seq)
    sigma = len(alpha)
    assert p.sigma == sigma and p.n == len(seq)
    assert bytes(p.sym_of_code[:sigma]) == alpha.tobytes()
    assert p.levels == (int(np.ceil(np.log2(sigma))) if sigma > 1 else 0)
    cnt = np.bincount(np.frombuffer(seq, dtype=np.uint8), minlength=256)
    a = list(range(sigma))
    for l, bits in enumerate(spine):
        mid = len(a) // 2
        for c in a:                                    # left-most node: starts at 0, bit = right half
            assert p.node_start[l][c] == 0 and p.node_id[l][c] == 0
            assert p.node_bit[l][c] == (1 if c >= a[mid] else 0)
        assert sum(int(cnt[alpha[c]]) for c in a) == len(bits)
        a = a[:mid]
    for l in range(p.levels):                          # every level: nodes tile the level exactly
        alive = [c for c in range(sigma) if p.depth[c] > l]
        assert p.level_len[l] == sum(int(p.cnt[c]) for c in alive)
    for c in range(sigma):
        assert p.C[c] == sum(int(p.cnt[k]) for k in range(c))
        assert p.depth[c] in (p.levels, p.levels - 1)


def test_error_codes_without_gpu():
    from hkcsa import _lib
    L = _lib.load()
    p = _lib.SsaPlan()
    assert L.hkcsa_ssa_plan_make(100, 0, C.byref(p)) == _lib.EINVAL
    assert b"bad argument" in L.hkcsa_last_error()
    assert L.hkcsa_ssa_plan_make(_lib.MAX_N + 1, 4, C.byref(p)) == _lib.ERANGE
    assert L.hkcsa_ssa_plan_make(1000, 8, C.byref(p)) == 0 and p.n_samples == 125
    with pytest.raises(_lib.HkcsaError):
        _lib.check(_lib.EINVAL)


def test_engine_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from hkcsa import engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.to_device_u8(b"banana")
    from csa.suffix_array import build_suffix_array
    with pytest.raises(RuntimeError):
        build_suffix_array("banana")


def test_views_list_semantics():
    from hkcsa import views
    t = torch.tensor([5, 3, 1, 0, 4, 2], dtype=torch.int32)
    s = views.DeviceSequence(t)
    assert len(s) == 6 and s[0] == 5 and s[-1] == 2 and s[1:3] == [3, 1]
    assert s == [5, 3, 1, 0, 4, 2] and not (s == [5, 3, 1, 0, 4, 3]) and s != [1]
    assert list(s) == s.tolist() == [5, 3, 1, 0, 4, 2]
    with pytest.raises(IndexError):
        s[6]
    assert views.int_sequence(t) == [5, 3, 1, 0, 4, 2] and isinstance(views.int_sequence(t), list)
    lz = views.LazyList(lambda: [1, 0, 1])
    assert lz == [1, 0, 1] and len(lz) == 3 and lz[0] == 1
    assert views.maybe_lazy(3, lambda: [7]) == [7]


def test_dropin_api_surface():
    """Same public names and signatures as the reference modules (SURVEY.md section 8b)."""
    import csa.suffix_array as sa
    import csa.bwt as bwt
    import csa.wavelet_tree as wt
    import csa.enhanced_fm_index as efm
    import csa.csa as csa_mod
    import utils.utils as uu
    import utils.data_loader as dl

    assert list(inspect.signature(sa.build_suffix_array).parameters) == ["text"]
    assert list(inspect.signature(sa.ksa).parameters) == ["T"]
    assert sa.optimized_ksa is sa.ksa
    assert list(inspect.signature(bwt.bwt_transform).parameters) == ["text", "suffix_array"]
    assert list(inspect.signature(uu.build_count).parameters) == ["text"]
    assert list(inspect.signature(uu.build_occ).parameters) == ["bwt"]
    assert list(inspect.signature(dl.load_text).parameters) == ["path", "size_limit"]
    for cls, methods in [
        (wt.SuccinctRankSelect, ["rank", "select"]),
        (wt.GolombRiceEncoder, ["compute_dynamic_m", "encode"]),
        (wt.WaveletTree, ["build_tree", "run_length_encode", "level_ordered_encode", "rank", "select",
                          "compress", "decompress"]),
        (efm.EnhancedFMIndex, ["find", "find_range", "rank"]),
        (csa_mod.FMIndex, ["precompute_rank", "backward_search", "find_pattern"]),
        (csa_mod.CompressedSuffixArray, ["locate"]),
    ]:
        for m in methods:
            assert callable(getattr(cls, m)), f"{cls.__name__}.{m}"
    assert list(inspect.signature(csa_mod.CompressedSuffixArray.__init__).parameters)[:3] == ["self", "text", "epsilon"]
    assert sa.text == "banana" and wt.text == "this is an example text"
    # integer restatement of the Golomb parameter needs no device
    enc = wt.GolombRiceEncoder.__new__(wt.GolombRiceEncoder)
    assert [enc.compute_dynamic_m(o, t) for o, t in [(1, 2), (1, 4), (1, 8), (3, 24), (1, 3), (1, 5), (0, 7)]] == \
        [1, 2, 3, 3, 1, 2, 1]


def test_golomb_m_matches_golden(golden):
    import csa.wavelet_tree as wt
    enc = wt.GolombRiceEncoder.__new__(wt.GolombRiceEncoder)
    for ones, total, m in golden.meta["_golomb_m"]:
        assert enc.compute_dynamic_m(ones, total) == m


def test_occ_table_plans_are_host_only():
    """hkcsa_occ_plan_make: layouts, sizes and argument checks (no GPU involved)."""
    from hkcsa import _lib
    L = _lib.load()
    p = _lib.OccPlan()
    n, sigma = 200_000_001, 97
    # layout 0, 32 rows per entry: [32 BWT bytes][sigma x u32], rows padded to 32 bytes
    assert L.hkcsa_occ_plan_make(n, sigma, 5, 0, C.byref(p)) == 0
    assert (p.rows, p.stride, p.layout, p.shift) == ((n >> 5) + 1, 448, 0, 5)
    assert p.blob_bytes >= p.rows * p.stride and p.blob_bytes % 256 == 0 and p.scratch_bytes > 0
    assert L.hkcsa_occ_plan_make(n, sigma, 6, 0, C.byref(p)) == 0 and p.stride == 480 and p.rows == (n >> 6) + 1
    # layout 1: one 8-byte entry per symbol and 32 rows, the BWT copy behind the entries
    assert L.hkcsa_occ_plan_make(n, sigma, 5, 1, C.byref(p)) == 0
    assert p.stride >= p.rows and p.stride % 4 == 0 and p.off_bwt >= 8 * sigma * p.stride
    assert p.blob_bytes >= p.off_bwt + n
    assert L.hkcsa_occ_plan_make(1, 1, 5, 1, C.byref(p)) == 0 and p.rows == 1
    # argument checks
    assert L.hkcsa_occ_plan_make(n, sigma, 4, 0, C.byref(p)) == _lib.EINVAL
    assert L.hkcsa_occ_plan_make(n, sigma, 6, 1, C.byref(p)) == _lib.EINVAL
    assert L.hkcsa_occ_plan_make(n, 0, 5, 0, C.byref(p)) == _lib.EINVAL
    assert L.hkcsa_occ_plan_make(n, 257, 5, 0, C.byref(p)) == _lib.EINVAL
    assert L.hkcsa_occ_plan_make(0, sigma, 5, 0, C.byref(p)) == _lib.ERANGE
    assert L.hkcsa_occ_plan_make(_lib.MAX_N + 1, sigma, 5, 0, C.byref(p)) == _lib.ERANGE


def test_peer_count_argument_checks_without_gpu():
    """hkcsa_count_batch_peers refuses malformed peer lists before touching the device."""
    from hkcsa import _lib
    L = _lib.load()
    wt = _plan(b"banana$")
    lo = (C.c_uint64 * 2)(0, 0)
    hi = (C.c_uint64 * 2)(0, 0)
    blob = C.create_string_buffer(64)
    args = (C.cast(blob, C.c_void_p), C.byref(wt), None, None, None, 0, None, None, 3, 0)
    assert L.hkcsa_count_batch_peers(*args, 0, lo, hi, None) == _lib.EINVAL          # no peers
    assert L.hkcsa_count_batch_peers(*args, 17, lo, hi, None) == _lib.EINVAL         # more than HKCSA_MAX_PEERS
    assert L.hkcsa_count_batch_peers(*args, 2, lo, hi, None) == _lib.EINVAL          # null offsets / null peer pointers
    occ = _lib.OccPlan()
    bad = (C.cast(blob, C.c_void_p), C.byref(wt), None, C.byref(occ), None, 0, None, None, 3, 0)
    assert L.hkcsa_count_batch_peers(*bad, 1, lo, hi, None) == _lib.EINVAL           # occ plan without its blob


def test_prof_class_names():
    from hkcsa import _lib
    L = _lib.load()
    assert L.hkcsa_prof_class_index(b"onesweep_u64") >= 0
    assert L.hkcsa_prof_class_index(b"bwt_gather") >= 0
    assert L.hkcsa_prof_class_index(b"no such kernel") == -1


def test_distributed_build_plan_is_host_only():
    """hkcsa_dsa_plan_make derives the round-0 prefix code and the id width from the byte histogram of the whole text
    (host memory only): the same inputs give the same plan on every rank; argument checks need no GPU."""
    from hkcsa import _lib
    L = _lib.load()
    assert L.hkcsa_dsa_state_bytes() == C.sizeof(C.c_uint64) * 512 and L.hkcsa_dsa_scratch_bytes(1 << 20) > (1 << 20) * 24

    def plan(hist, n, wide=0):
        h = np.zeros(256, dtype=np.uint64)
        for k, v in hist.items():
            h[k] = v
        p = _lib.DsaPlan()
        rc = L.hkcsa_dsa_plan_make(h.ctypes.data_as(C.POINTER(C.c_uint64)), n, wide, C.byref(p))
        return rc, p

    rc, dna = plan({65: 25, 67: 25, 71: 25, 84: 25, 36: 1}, 101)
    assert rc == 0 and dna.sigma == 5 and dna.bits0 % 8 == 0 and 16 <= dna.bits0 <= 64 and dna.passes0 == dna.bits0 // 8
    assert dna.wide == 0 and dna.k0 >= 1 and dna.b_fixed == 3
    codes = [(dna.code[c], dna.len[c]) for c in (256, 36, 65, 67, 71, 84)]       # past-the-end, then bytes in order
    streams = [format(c, "b").zfill(l) for c, l in codes]
    assert streams == sorted(streams) and len(set(streams)) == 6                   # order-preserving ...
    assert not any(a != b and b.startswith(a) for a in streams for b in streams)   # ... and prefix-free
    assert [dna.fixed_code[c] for c in (36, 65, 67, 71, 84)] == [1, 2, 3, 4, 5] and dna.fixed_code[66] == 0
    rc2, again = plan({65: 25, 67: 25, 71: 25, 84: 25, 36: 1}, 101)
    assert bytes(again) == bytes(dna)
    assert plan({97: 10}, (1 << 32) - 2)[1].wide == 0 and plan({97: 10}, (1 << 32) - 1)[1].wide == 1
    assert plan({97: 10}, 100, wide=1)[1].wide == 1
    assert plan({97: 10}, (1 << 40) + 1)[0] == _lib.ERANGE
    one = plan({97: 1000}, 1000)[1]
    assert one.sigma == 1 and one.bits0 >= 16
    # argument checks of the device entry points come before any CUDA call
    st = C.create_string_buffer(L.hkcsa_dsa_state_bytes())
    assert L.hkcsa_dsa_ext_round(st, None) == _lib.EINVAL                           # state not initialised by _begin
    assert L.hkcsa_dsa_working_set(st) == 0 and L.hkcsa_dsa_slice(st) is None
    cuts = (C.c_uint32 * 3)(0, 10, 65535)                                          # does not span every bucket
    z = (C.c_uint64 * 2)(0, 0)
    assert L.hkcsa_dsa_pack_exchange(1, C.byref(dna), 0, 0, 2, cuts, z, z, z, 1, None) == _lib.EINVAL
    assert L.hkcsa_dsa_pack_exchange(1, C.byref(dna), 0, 0, 9, cuts, z, z, z, 1, None) == _lib.EINVAL
    assert L.hkcsa_ranges_push_peers(1, 1, 5, 0, 17, z, 0, None) == _lib.EINVAL
    assert L.hkcsa_ranges_push_peers(None, None, 0, 0, 1, z, 0, None) == 0          # empty slice: nothing to do
    assert L.hkcsa_entropy_scratch_bytes(1000) > 1000 * 9 and L.hkcsa_rrr_scratch_bytes(960 * 100) >= 100 * 24
    out = (C.c_double * 5)()
    assert L.hkcsa_entropy_from_sa(None, 10, None, 0, out, None, 0, None) == _lib.EINVAL       # k = 0 is the histogram's job
    assert L.hkcsa_entropy_from_sa(None, 3, None, 5, out, None, 0, None) == 0 and list(out) == [0.0] * 5   # n <= k -> 0


def test_distributed_plan_id_width_and_size_limit():
    """Suffix ids stay 32-bit up to 2^32 - 2 symbols (one id value is kept free) and widen at 2^32 - 1; the build
    takes texts up to 2^40 symbols and refuses one more with ERANGE."""
    from hkcsa import _lib
    L = _lib.load()
    h = np.zeros(256, dtype=np.uint64)
    h[97] = 10

    def make(n):
        p = _lib.DsaPlan()
        return L.hkcsa_dsa_plan_make(h.ctypes.data_as(C.POINTER(C.c_uint64)), n, 0, C.byref(p)), p

    assert _lib.DSA_MAX_N32 == (1 << 32) - 2
    for n, rc, wide in (((1 << 32) - 2, 0, 0), ((1 << 32) - 1, 0, 1), (1 << 40, 0, 1)):
        got_rc, p = make(n)
        assert (got_rc, p.wide, p.n) == (rc, wide, n), n
    assert make((1 << 40) + 1)[0] == _lib.ERANGE and b"2^40" in L.hkcsa_last_error()


def test_multi_slice_descriptor_argument_checks_without_gpu():
    """hkcsa_multi_desc_build refuses a bad slice count, n > 2^40, slice lengths that differ from their plans and a row
    of suffix 0 outside [0, n) -- each before any CUDA call (none of the pointers is a device address)."""
    from hkcsa import _lib
    L = _lib.load()
    parts = [b"banana", b"$abc"]
    plans = [_plan(x) for x in parts]
    ssa = []
    for x in parts:
        sp = _lib.SsaPlan()
        assert L.hkcsa_ssa_plan_make_slice(len(x), 4, 1, C.byref(sp)) == 0
        ssa.append(sp)
    n = sum(len(x) for x in parts)
    fake = [0x1000, 0x2000]

    def build(S, starts, with_ssa=True, row0=0, plan_list=plans):
        k = max(S, 1)
        blobs = (C.c_void_p * k)(*(fake * k)[:k])
        pl = (C.POINTER(_lib.WtPlan) * k)(*[C.pointer(plan_list[i % 2]) for i in range(k)])
        st = (C.c_uint64 * len(starts))(*starts)
        sb = (C.c_void_p * k)(*(fake * k)[:k]) if with_ssa else None
        sp = (C.POINTER(_lib.SsaPlan) * k)(*[C.pointer(ssa[i % 2]) for i in range(k)]) if with_ssa else None
        return L.hkcsa_multi_desc_build(S, blobs, pl, st, sb, sp, row0, C.c_void_p(0x3000), None)

    assert build(0, [0]) == _lib.EINVAL
    assert build(9, [0] + [n] * 9) == _lib.EINVAL and b"slices" in L.hkcsa_last_error()
    assert build(2, [0, 6, (1 << 40) + 1]) == _lib.ERANGE and b"2^40" in L.hkcsa_last_error()
    assert build(2, [0, 5, n]) == _lib.EINVAL and b"plan length" in L.hkcsa_last_error()
    assert build(2, [0, 6, n], plan_list=plans[::-1]) == _lib.EINVAL
    for row0 in (n, n + 1, (1 << 64) - 1):
        assert build(2, [0, 6, n], row0=row0) == _lib.EINVAL and b"row0" in L.hkcsa_last_error(), row0
    assert build(2, [0, 6, n], with_ssa=False, row0=n) == _lib.EINVAL and b"row0" in L.hkcsa_last_error()


def test_pack_patterns_host_fast_and_slow_paths_agree():
    """One join + one encode for a list of latin-1 str patterns; bytes / mixed lists pattern by pattern: same CSR."""
    from hkcsa import engine
    pats = ["ana", "", "banana", "caf\xe9", "x" * 300]
    flat, off = engine.pack_patterns_host(pats)
    assert flat == "".join(pats).encode("latin-1") and off.tolist() == [0, 3, 3, 9, 13, 313] and off.dtype == np.int64
    as_bytes = [p.encode("latin-1") for p in pats]
    for variant in (as_bytes, [pats[0], as_bytes[1], bytearray(as_bytes[2]), pats[3], memoryview(as_bytes[4])]):
        f2, o2 = engine.pack_patterns_host(variant)
        assert f2 == flat and np.array_equal(o2, off)
    f0, o0 = engine.pack_patterns_host([])
    assert f0 == b"" and o0.tolist() == [0]
    with pytest.raises(UnicodeEncodeError):              # beyond latin-1: the drop-in layer turns it into a miss
        engine.pack_patterns_host(["ab", "sn\u2603w"])


def test_symbol_map_ascii_latin1_and_wide_texts():
    """ASCII text: nothing is encoded (host_bytes hands the str itself to the staged copy); latin-1: one encode;
    beyond latin-1: order-preserving re-coding (the reference compares code points, csa/suffix_array.py:132)."""
    from hkcsa import engine
    text = "GATTACA" * 1000
    m = engine.SymbolMap(text, extra="$")
    assert m.identity and m.host_bytes(text) is text and m.encode("$") == b"$" and m.encode("\u2603") is None
    lat = "caf\xe9" * 10
    m2 = engine.SymbolMap(lat, extra="$")
    assert m2.identity and m2.host_bytes(lat) == lat.encode("latin-1")
    wide = "\u03b1\u03b2\u03b1\u03b3$"
    m3 = engine.SymbolMap(wide, extra="$")
    assert not m3.identity and m3.host_bytes(wide) == m3.encode(wide)
    enc = m3.encode(wide)
    assert [m3.symbol(b) for b in enc] == list(wide) and m3.decode(enc) == wide
    assert sorted(set(enc)) == list(range(len(set(wide)))) and m3.encode("\u03b4") is None
    order = sorted(set(wide))
    assert [m3.encode(c)[0] for c in order] == list(range(len(order)))      # code points keep their order
