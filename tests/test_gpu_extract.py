"""Extract (csrc/extract.cu): inverse-SA samples from the sampled SA, batched text extraction by LF walks, and the
drop-in CompressedSuffixArray.extract / save / load built on them.  The argument checks of the two C entry points
run without a GPU; everything else is marked gpu and compared with the CPU oracle or the generated text."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O

gpu = pytest.mark.gpu


# ------------------------------------------------------------------ texts (all end with a unique '$')
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
    alpha = np.array([b for b in range(256) if b != 0x24], dtype=np.uint8)
    rng = np.random.RandomState(seed)
    body = alpha[rng.randint(0, alpha.size, size=n)]
    body[: alpha.size] = alpha                      # every one of the 255 symbols occurs
    return body.tobytes()


TEXTS = {
    "sigma1_n1": lambda: b"$",
    "sigma2": lambda: b"a" * 777 + b"$",
    "sigma5_dna": lambda: O.gen_text(O.DNA4, 3, 5000).tobytes() + b"$",
    "sigma97_eng": lambda: O.gen_text(O.ENG96, 4, 5000).tobytes() + b"$",
    "sigma256": lambda: _all_bytes(20_000) + b"$",
    "periodic": lambda: b"abcab" * 999 + b"$",
    "fibonacci": lambda: _fib(10_000).encode() + b"$",
    "runs": lambda: _runs(30_000) + b"$",
    "eng_300k": lambda: O.gen_text(O.ENG96, 42, 300_000).tobytes() + b"$",
    "dna_300k": lambda: O.gen_text(O.DNA4, 43, 300_000).tobytes() + b"$",
}
LF_MODES = ["wt", "occ0_shift5", "occ0_shift6", "occ1"]


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _index(E, text: bytes, rate: int, mode: str = "wt"):
    idx = E.DeviceIndex(E.to_device_u8(text), sa_sample_rate=rate)
    if mode != "wt":
        layout, shift = (1, 5) if mode == "occ1" else (0, int(mode[-1]))
        idx.build_occ_table(shift, layout=layout)
    return idx


def _extract_host(idx, begin, end, mode="wt"):
    import torch
    b = torch.tensor(begin, dtype=torch.int64, device=idx.device)
    e = torch.tensor(end, dtype=torch.int64, device=idx.device)
    off, out = idx.extract_batch(b, e, use_occ_table=(mode != "wt"))
    off, out = off.cpu().numpy(), out.cpu().numpy().tobytes()
    return [out[off[q]:off[q + 1]] for q in range(len(begin))]


# ------------------------------------------------------------------ C-ABI argument checks (no GPU needed)
def _wt_plan(seq: bytes):
    from hkcsa import _lib
    hist = np.bincount(np.frombuffer(seq, dtype=np.uint8), minlength=256).astype(np.uint64)
    p = _lib.WtPlan()
    assert _lib.load().hkcsa_wt_plan_from_hist(hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(p)) == 0
    return p


def test_isa_samples_argument_checks_without_gpu():
    from hkcsa import _lib
    L = _lib.load()
    fake = C.c_void_p(0x1000)                       # never dereferenced: every check below fails first
    p = _lib.SsaPlan()
    assert L.hkcsa_ssa_plan_make(1000, 8, C.byref(p)) == 0
    assert L.hkcsa_isa_samples(None, C.byref(p), fake, None) == _lib.EINVAL            # null blob
    assert L.hkcsa_isa_samples(fake, None, fake, None) == _lib.EINVAL                  # null plan
    assert L.hkcsa_isa_samples(fake, C.byref(p), None, None) == _lib.EINVAL            # null output
    bad = _lib.SsaPlan.from_buffer_copy(bytes(p))
    bad.rate = 0
    assert L.hkcsa_isa_samples(fake, C.byref(bad), fake, None) == _lib.EINVAL          # rate 0
    sl = _lib.SsaPlan()
    assert L.hkcsa_ssa_plan_make_slice(1000, 8, 120, C.byref(sl)) == 0                 # 120 marks != ceil(1000 / 8)
    assert L.hkcsa_isa_samples(fake, C.byref(sl), fake, None) == _lib.EINVAL
    assert b"slice" in L.hkcsa_last_error()


def test_extract_argument_checks_without_gpu():
    from hkcsa import _lib
    L = _lib.load()
    fake = C.c_void_p(0x1000)
    wt = _wt_plan(b"banana$")
    occ = _lib.OccPlan()
    assert L.hkcsa_occ_plan_make(7, wt.sigma, 5, 1, C.byref(occ)) == 0
    need = L.hkcsa_extract_scratch_bytes(3)
    assert need >= 4 * 8 and L.hkcsa_extract_scratch_bytes(1 << 20) > need

    def call(wt_blob=fake, wtp=C.byref(wt), ob=None, op=None, isa=fake, rate=4, R=3, out=fake, scratch=fake, nbytes=need):
        return L.hkcsa_extract(wt_blob, wtp, ob, op, isa, rate, fake, fake, fake, R, out, scratch, nbytes, None)

    assert call(wt_blob=None) == _lib.EINVAL
    assert call(wtp=None) == _lib.EINVAL
    assert call(isa=None) == _lib.EINVAL
    assert call(rate=0) == _lib.EINVAL
    assert call(ob=fake) == _lib.EINVAL                          # occ blob without its plan
    assert call(op=C.byref(occ)) == _lib.EINVAL                  # occ plan without its blob
    other = _lib.OccPlan()
    assert L.hkcsa_occ_plan_make(8, wt.sigma, 5, 1, C.byref(other)) == 0
    assert call(ob=fake, op=C.byref(other)) == _lib.EINVAL       # occ plan of another index
    assert call(out=None) == _lib.EINVAL
    assert call(scratch=None) == _lib.EINVAL
    assert call(nbytes=need - 1) == _lib.ESCRATCH
    assert call(R=0, out=None, scratch=None) == _lib.OK          # nothing to do: no device work


def test_symbol_map_from_code_points():
    from hkcsa.engine import SymbolMap
    text = "aĀbā$"
    m = SymbolMap(text, extra="$")
    back = SymbolMap.from_code_points(m.back)
    assert back.encode(text) == m.encode(text) and back.decode(m.encode(text)) == text
    ident = SymbolMap.from_code_points([])
    assert ident.identity and ident.decode(b"ab\xe9") == "abé"


# ------------------------------------------------------------------ inverse-SA samples
@gpu
@pytest.mark.parametrize("rate", [1, 2, 3, 7, 16, 64])
@pytest.mark.parametrize("n", [1, 50, 1000, 4097])
def test_isa_samples_match_oracle(E, rate, n):
    text = (O.gen_text(O.DNA4, 11 + n, n - 1).tobytes() if n > 1 else b"") + b"$"
    idx = _index(E, text, rate)
    isa = idx.isa_samples().cpu().numpy()
    S = -(-n // rate)
    assert isa.size == S + 1
    inv = np.argsort(O.build_suffix_array(text))
    assert np.array_equal(isa[:S], inv[np.arange(S) * rate])
    assert isa[S] == isa[0]


# ------------------------------------------------------------------ whole text
@gpu
@pytest.mark.parametrize("mode", LF_MODES)
@pytest.mark.parametrize("name", list(TEXTS))
def test_whole_text_extract(E, name, mode):
    text = TEXTS[name]()
    for rate in (1, 6, 32) if len(text) < 50_000 else (6,):
        idx = _index(E, text, rate, mode)
        assert idx.invertible
        got = idx.extract(0, len(text), use_occ_table=(mode != "wt"))
        assert got.cpu().numpy().tobytes() == text, (name, mode, rate)


# ------------------------------------------------------------------ ranges
@gpu
@pytest.mark.parametrize("mode", ["wt", "occ1", "occ0_shift6"])
@pytest.mark.parametrize("rate", [1, 5, 16, 200])
def test_range_batches(E, mode, rate):
    text = O.gen_text(O.ENG96, 9, 3000).tobytes() + b"$"
    n = len(text)
    idx = _index(E, text, rate, mode)
    rng = np.random.RandomState(rate)
    b = rng.randint(0, n + 1, size=500)
    e = np.minimum(n, b + rng.randint(0, 3 * rate + 2, size=500))
    extra = [(0, 0), (n, n), (n - 1, n), (0, n), (n - 7, n), (rate - 1, rate + 1), (rate, 2 * rate), (17, 17),
             (max(0, n - rate - 3), n - 1)]
    begin = list(b) + [x for x, _ in extra] + list(range(n))
    end = list(e) + [y for _, y in extra] + list(range(1, n + 1))      # every length-1 range
    got = _extract_host(idx, begin, end, mode)
    for q, (x, y) in enumerate(zip(begin, end)):
        assert got[q] == text[x:y], (q, x, y)


@gpu
def test_invalid_ranges_are_refused_and_clamped_on_device(E):
    import torch
    from hkcsa import _lib
    text = O.gen_text(O.DNA4, 8, 999).tobytes() + b"$"
    n = len(text)
    idx = _index(E, text, 7)
    for b, e in [(-1, 5), (5, 4), (0, n + 1)]:
        with pytest.raises(ValueError, match="begin <= end"):
            _extract_host(idx, [b], [e])
    # straight through the C-ABI: out-of-range requests are clamped to [0, n] and to their own output slice
    begin = torch.tensor([-50, 990, 10, 300], dtype=torch.int64, device="cuda")
    end = torch.tensor([20, 5000, 5, 310], dtype=torch.int64, device="cuda")
    out_off = torch.tensor([0, 30, 40, 41, 51], dtype=torch.int64, device="cuda")   # slices of 30, 10, 1, 10 bytes
    out = torch.full((51 + 64,), 0xEE, dtype=torch.uint8, device="cuda")
    L = _lib.load()
    nbytes = L.hkcsa_extract_scratch_bytes(4)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    isa = idx.isa_samples()
    _lib.check(L.hkcsa_extract(idx.wt.blob.data_ptr(), C.byref(idx.wt.plan), None, None, isa.data_ptr(), 7,
                               begin.data_ptr(), end.data_ptr(), out_off.data_ptr(), 4, out.data_ptr(),
                               scratch.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream))
    got = out.cpu().numpy().tobytes()
    assert got[0:20] == text[0:20] and got[20:30] == b"\xee" * 10        # [-50, 20) -> [0, 20)
    assert got[30:40] == text[990:1000]                                  # [990, 5000) -> [990, n)
    assert got[40:41] == b"\xee"                                         # end < begin: nothing
    assert got[41:51] == text[300:310]
    assert got[51:] == b"\xee" * 64                                      # nothing past the last slice


# ------------------------------------------------------------------ a loaded index gives the text back
@gpu
@pytest.mark.parametrize("mode", ["wt", "occ1"])
def test_loaded_index_extracts_the_text(E, tmp_path, mode):
    text = O.gen_text(O.ENG96, 21, 200_000).tobytes() + b"$"
    idx = _index(E, text, 9)
    path = str(tmp_path / "idx.npz")
    idx.save(path, compressed=True)
    del idx
    back = E.DeviceIndex.load(path)
    assert back.text is None and back.sa is None and back.bwt is None
    if mode == "occ1":                         # a replica is handed the BWT to build its Occ table from
        back.build_occ_table(5, bwt=E.to_device_u8(O.bwt_transform(text, O.build_suffix_array(text))), layout=1)
    assert back.extract(0, back.n, use_occ_table=(mode == "occ1")).cpu().numpy().tobytes() == text
    assert _extract_host(back, [1000, 5], [1100, 5], mode) == [text[1000:1100], b""]


# ------------------------------------------------------------------ invertibility
@gpu
def test_invertible_only_when_lf_inverts_the_suffix_order(E):
    good = _index(E, b"a$b$", 2)
    assert good.invertible
    assert good.extract(0, 4).cpu().numpy().tobytes() == b"a$b$"
    for text in (b"ab$ab$", b"mississippi$" * 40 + b"$"):
        idx = _index(E, text, 3)
        assert not idx.invertible
        with pytest.raises(ValueError, match="sentinel"):
            idx.extract(0, len(text))


# ------------------------------------------------------------------ drop-in CompressedSuffixArray
CSA_TEXTS = {
    "ascii": O.gen_text(O.ENG96, 31, 20_000).tobytes().decode("latin-1"),
    "latin1": "café naïve über " * 700,
    "recoded": "Āāab中文-" * 900,
    "bytes": bytes(range(256)).replace(b"$", b"") * 40,
}


@gpu
@pytest.mark.parametrize("name", list(CSA_TEXTS))
def test_csa_extract_slices(cuda, name, tmp_path):
    from csa.csa import CompressedSuffixArray
    text = CSA_TEXTS[name]
    csa = CompressedSuffixArray(text)
    m = len(text)
    bounds = [(0, m), (3, 50), (-10, None), (None, 7), (-m - 5, 4), (m - 3, m + 100), (40, 20), (m, m), (0, 0),
              (-1, -1), (5, -5)]
    for a, b in bounds:
        got = csa.extract(a, b)
        assert type(got) is type(text) and got == text[a:b], (a, b)
    pairs = [(k, k + 33) for k in range(0, m, 997)]
    assert csa.extract_batch(pairs) == [text[a:b] for a, b in pairs]
    # save -> load: a query-only object that holds no text and answers like the built one
    path = str(tmp_path / "csa.npz")
    csa.save(path)
    back = CompressedSuffixArray.load(path)
    assert back._text is None
    pats = [text[100:104], text[7:9], text[-5:], text[:1]]
    assert [back.count(p) for p in pats] == [csa.count(p) for p in pats]
    assert [back.locate(p) for p in pats] == [csa.locate(p) for p in pats]
    assert back.extract(-300, -2) == text[-300:-2]
    assert back.sa_sample_rate == csa.sa_sample_rate and back.epsilon == csa.epsilon
    assert back.index_bytes() == csa.index_bytes()
    assert back.space_report()["n"] == csa.space_report()["n"]
    assert back.text == text and type(back.text) is type(text)


@gpu
def test_csa_text_holding_the_sentinel(cuda, tmp_path):
    from csa.csa import CompressedSuffixArray
    ok = CompressedSuffixArray("a$b")                 # '$' inside, yet LF still inverts the suffix order
    assert ok.extract(0, 3) == "a$b"
    bad = CompressedSuffixArray("mississippi$" * 40)
    with pytest.raises(ValueError, match="sentinel"):
        bad.extract(0, 5)
    assert bad.locate("ssi") == [m for m in range(480) if ("mississippi$" * 40).startswith("ssi", m)]
    path = str(tmp_path / "bad.npz")
    bad.save(path)
    with pytest.raises(ValueError, match="suffix array"):
        CompressedSuffixArray.load(path)


# ------------------------------------------------------------------ full size
@gpu
def test_full_size_dna_extract(E):
    import torch
    n = 100_000_000
    text = torch.cat([E.gen_text(E.DNA4, 43, n), torch.tensor([0x24], dtype=torch.uint8, device="cuda")])
    idx = E.DeviceIndex(text, sa_sample_rate=6, keep_sa=False)
    idx.bwt = None
    assert torch.equal(idx.extract(0, n + 1), text)
    g = torch.Generator(device="cuda").manual_seed(7)
    R, m = 1_000_000, 64
    begin = torch.randint(0, n + 1 - m, (R,), generator=g, device="cuda", dtype=torch.int64)
    off, out = idx.extract_batch(begin, begin + m)
    assert torch.equal(off, torch.arange(R + 1, device="cuda", dtype=torch.int64) * m)
    want = text[begin[:, None] + torch.arange(m, device="cuda")]
    assert torch.equal(out.view(R, m), want)
