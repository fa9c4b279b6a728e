"""Extract over the sliced index a distributed build leaves behind (hkcsa.dist_sa.MultiSliceIndex): inverse-SA samples
from the slices' sampled suffix arrays, and text ranges by LF walks that hop across slices with the exact step.

The texts include ones whose last symbol occurs earlier too ("mississippi$" * k, a second '$', an English-like text
whose last letter recurs).  There the plain LF step does not invert the suffix order (the single-GPU extract refuses
such an index), so these tests show that the sliced walk gives the text back on every text.  The indexes are built
as in test_gpu_multi_slice.py: over the oracle's suffix array and BWT cut at given rows, over what
emulate_distributed_suffix_array returns, through replicate_sliced_index, and at the sizes of the distributed
envelope (test_gpu_dist_envelope.py), checked there against the exact ISA of tests/device_reference.py."""
import json
import time

import numpy as np
import pytest
import torch

import device_reference as R
from test_gpu_dist_envelope import CASES, GB, RATE, _peak_bytes
from test_gpu_multi_slice import DIST_TEXTS, LOCATE_TEXTS, _ms_from_sa, _oracle

pytestmark = pytest.mark.gpu

TEXTS = {**LOCATE_TEXTS, "dollar": b"$", "a$": b"a$"}
NOT_INVERTIBLE = {"mississippi_k", "mississippi_k_dollar", "ab$ab$", "a$b$a$"}


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _rate(rate, n):
    return n + 5 if rate == "over_n" else rate


def _occ_at_row0(sa, bwt) -> int:
    """occ(bwt[row0], row0) from the oracle: > 0 exactly when the plain LF step is wrong at the row of suffix 0."""
    row0 = int(np.flatnonzero(sa == 0)[0])
    return int((bwt[:row0] == bwt[row0]).sum())


def _extract_host(ms, begin, end):
    b = torch.tensor(begin, dtype=torch.int64, device="cuda")
    e = torch.tensor(end, dtype=torch.int64, device="cuda")
    off, out = ms.extract_batch(b, e)
    off, out = off.cpu().numpy(), out.cpu().numpy().tobytes()
    return [out[off[q]:off[q + 1]] for q in range(len(begin))]


def _check_text(ms, text: bytes, rate: int, seed: int = 0):
    """The whole text, every length-1 range, every range across a sample boundary, the last stretch, empty ranges and
    random ranges, each against the text's bytes."""
    n = len(text)
    assert ms.extract(0, n).cpu().numpy().tobytes() == text
    rng = np.random.RandomState(seed)
    rb = rng.randint(0, n + 1, size=300)
    re_ = np.minimum(n, rb + rng.randint(0, 3 * rate + 2, size=300))
    pairs = [(i, i + 1) for i in range(n)]                                       # every length-1 range
    pairs += [(k * rate - 1, min(n, k * rate + 1)) for k in range(1, -(-n // rate))]   # across every sample boundary
    pairs += [(max(0, n - rate - 1), n), (0, 0), (n, n), (n // 2, n // 2)]        # the last stretch, empty ranges
    pairs += list(zip(rb.tolist(), re_.tolist()))
    got = _extract_host(ms, [a for a, _ in pairs], [b for _, b in pairs])
    for q, (a, b) in enumerate(pairs):
        assert got[q] == text[a:b], (q, a, b)


def test_test_texts_exercise_the_exact_step():
    """The texts listed as not invertible really have occ(bwt[row0], row0) > 0, the others a unique last symbol."""
    for name, text in TEXTS.items():
        sa, bwt = _oracle(text)
        assert (_occ_at_row0(sa, bwt) > 0) == (name in NOT_INVERTIBLE), name


# ------------------------------------------------------------------ inverse samples
@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("parts", [1, 2, 3, 8])
@pytest.mark.parametrize("rate", [1, 3, 32, "over_n"])
@pytest.mark.parametrize("name", list(TEXTS))
def test_multi_isa_samples(E, name, rate, parts, wide):
    """isa[k] == argsort(sa)[k * rate] for k < ceil(n / rate), isa[S] == isa[0]; 1-8 slices, empty ones included."""
    text = TEXTS[name]
    n = len(text)
    rate = _rate(rate, n)
    sa, bwt = _oracle(text)
    ms = _ms_from_sa(text, sa, bwt, [n * r // parts for r in range(parts + 1)], rate, wide)
    isa = ms.isa_samples()
    assert isa.dtype == torch.int64 and ms.isa_samples() is isa                  # cached
    isa = isa.cpu().numpy()
    S = -(-n // rate)
    assert isa.size == S + 1
    inv = np.argsort(sa)
    assert np.array_equal(isa[:S], inv[np.arange(S) * rate]) and isa[S] == isa[0]


# ------------------------------------------------------------------ whole text and ranges
@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("parts", [1, 2, 3, 8])
@pytest.mark.parametrize("rate", [1, 3, 32, "over_n"])
@pytest.mark.parametrize("name", list(TEXTS))
def test_multi_extract_ranges(E, name, rate, parts, wide):
    text = TEXTS[name]
    n = len(text)
    rate = _rate(rate, n)
    sa, bwt = _oracle(text)
    ms = _ms_from_sa(text, sa, bwt, [n * r // parts for r in range(parts + 1)], rate, wide)
    _check_text(ms, text, rate, seed=parts * 100 + (rate % 97))


@pytest.mark.parametrize("edge", ["first", "last"])
@pytest.mark.parametrize("rate", [3, 32])
def test_multi_extract_with_row0_at_a_slice_edge(E, edge, rate):
    """The row of suffix 0 as the first row of a slice and as the last, with '$' in the slices before it: the step at
    row0 goes to C['$'], not past the '$' rows of the earlier slices."""
    text = b"mississippi$" * 60 + b"$"
    sa, bwt = _oracle(text)
    n = len(text)
    assert _occ_at_row0(sa, bwt) > 0
    row0 = int(np.flatnonzero(sa == 0)[0])
    cut = row0 if edge == "first" else row0 + 1
    cuts = sorted({0, n // 5, cut, (4 * n) // 5, n})
    ms = _ms_from_sa(text, sa, bwt, cuts, rate, wide=False)
    s = cuts.index(cut)
    assert ms.starts[s] == cut
    _check_text(ms, text, rate)


# ------------------------------------------------------------------ over the emulated distributed build
@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("name", list(DIST_TEXTS))
def test_multi_extract_over_the_distributed_build(E, name, wide):
    from hkcsa import dist_sa
    text, parts = DIST_TEXTS[name]
    n = len(text)
    d = E.to_device_u8(text)
    bounds = [n * r // parts for r in range(parts + 1)]
    slices = dist_sa.emulate_distributed_suffix_array([d[bounds[r]:bounds[r + 1]].clone() for r in range(parts)],
                                                      wide=wide)
    ms = dist_sa.MultiSliceIndex(n, [{"bwt": sl.bwt, "sa": sl.sa} for sl in slices], sa_sample_rate=32)
    sa, _ = _oracle(text)
    S = -(-n // 32)
    assert np.array_equal(ms.isa_samples().cpu().numpy(), np.argsort(sa)[np.r_[np.arange(S) * 32, 0]])
    assert torch.equal(ms.extract(0, n), d)
    rng = np.random.RandomState(n % 1000)
    b = rng.randint(0, n + 1, size=3000)
    e = np.minimum(n, b + rng.randint(0, 200, size=3000))
    got = _extract_host(ms, b.tolist(), e.tolist())
    for q in range(3000):
        assert got[q] == text[b[q]:e[q]], (q, b[q], e[q])


def test_replicated_sliced_index_extracts_the_text(E):
    """replicate_sliced_index (one NCCL rank in this process): the replica's index extracts the whole text."""
    import torch.distributed as dist
    from hkcsa import dist_sa
    text = b"mississippi$" * 2_000
    sl, = dist_sa.emulate_distributed_suffix_array([E.to_device_u8(text)])
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        ms = dist_sa.replicate_sliced_index(sl, sa_sample_rate=32)
    finally:
        dist.destroy_process_group()
    assert ms.extract(0, len(text)).cpu().numpy().tobytes() == text
    assert _extract_host(ms, [5, 23_990], [40, 24_000]) == [text[5:40], text[23_990:]]


# ------------------------------------------------------------------ refusals and clamping
def test_refusals_and_device_clamping(E):
    from hkcsa import _lib, dist_sa
    text = b"mississippi$" * 80
    n = len(text)
    sa, bwt = _oracle(text)
    ms = _ms_from_sa(text, sa, bwt, [0, 300, 700, n], 7, wide=False)
    for b, e in [(-1, 5), (5, 4), (0, n + 1)]:
        with pytest.raises(ValueError, match="begin <= end"):
            _extract_host(ms, [b], [e])
    bare = dist_sa.MultiSliceIndex(n, [{"bwt": torch.from_numpy(bwt[:500].copy()).cuda()},
                                       {"bwt": torch.from_numpy(bwt[500:].copy()).cuda()}])
    for call in (bare.isa_samples, lambda: bare.extract(0, 5), lambda: _extract_host(bare, [0], [5])):
        with pytest.raises(ValueError, match="without a sampled suffix array"):
            call()
    # straight through the C-ABI: out-of-range requests are clamped to [0, n] and to their own output slice
    begin = torch.tensor([-50, 950, 10, 300], dtype=torch.int64, device="cuda")
    end = torch.tensor([20, 5000, 5, 310], dtype=torch.int64, device="cuda")
    out_off = torch.tensor([0, 30, 40, 41, 51], dtype=torch.int64, device="cuda")   # slices of 30, 10, 1, 10 bytes
    out = torch.full((51 + 64,), 0xEE, dtype=torch.uint8, device="cuda")
    L = _lib.load()
    nbytes = L.hkcsa_extract_scratch_bytes(4)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    isa = ms.isa_samples()
    _lib.check(L.hkcsa_multi_extract(ms.desc.data_ptr(), n, 7, isa.data_ptr(), begin.data_ptr(), end.data_ptr(),
                                     out_off.data_ptr(), 4, out.data_ptr(), scratch.data_ptr(), nbytes,
                                     torch.cuda.current_stream().cuda_stream))
    got = out.cpu().numpy().tobytes()
    assert got[0:20] == text[0:20] and got[20:30] == b"\xee" * 10        # [-50, 20) -> [0, 20)
    assert got[30:40] == text[950:960]                                   # [950, 5000) -> [950, 960): its 10 bytes
    assert got[40:41] == b"\xee"                                         # end < begin: nothing
    assert got[41:51] == text[300:310]
    assert got[51:] == b"\xee" * 64                                      # nothing past the last slice


# ------------------------------------------------------------------ the distributed envelope
def _check_ranges_on_device(ms, text, b, e, what):
    off, out = ms.extract_batch(b, e)
    ln = e - b
    assert torch.equal(off[1:] - off[:-1], ln), what
    first = torch.repeat_interleave(b, ln)
    pos = first + torch.arange(out.numel(), device=b.device) - torch.repeat_interleave(off[:-1], ln)
    assert torch.equal(out, text[pos]), what


@pytest.mark.parametrize("case", ["eng_2g", "dna_wide", "mississippi"])
def test_multi_extract_at_scale(E, case):
    """The three envelope cases: inverse samples against the exact ISA, the whole text, 10^5 random ranges and ranges
    around every block cut and at the end of the text, each compared on the device."""
    from hkcsa import dist_sa
    n, make, frac, wide, _, skew = CASES[case]
    dev = torch.device("cuda", 0)
    torch.cuda.empty_cache()
    need = _peak_bytes(n, bool(wide), skew)
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need:
        pytest.skip(f"{case}: needs {need / GB:.1f} GiB of device memory, {free / GB:.1f} GiB free")
    t_case = time.perf_counter()
    torch.cuda.reset_peak_memory_stats(dev)
    text = make(E, n, dev)
    cuts = [int(n * f) for f in frac]
    world = len(cuts) - 1
    slices = dist_sa.emulate_distributed_suffix_array([text[cuts[r]:cuts[r + 1]] for r in range(world)], wide=wide)
    sa = torch.cat([sl.sa_int64() for sl in slices])
    isa = R.check_suffix_array(text, sa)
    del sa
    ms = dist_sa.MultiSliceIndex(n, [{"bwt": sl.bwt, "sa": sl.sa} for sl in slices], sa_sample_rate=RATE)
    del slices
    ctx = f"{case}: n={n}, ranks={world}"
    S = -(-n // RATE)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = ms.isa_samples()
    torch.cuda.synchronize()
    t_isa = time.perf_counter() - t0
    want = isa[torch.arange(S, device=dev) * RATE].to(torch.int64)
    assert torch.equal(got[:S], want) and int(got[S]) == int(isa[0]), f"{ctx}: inverse samples"
    del isa, want
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    whole = ms.extract(0, n)
    torch.cuda.synchronize()
    t_whole = time.perf_counter() - t0
    assert torch.equal(whole, text), f"{ctx}: whole text"
    del whole
    g = torch.Generator(device=dev).manual_seed(n)
    b = torch.randint(0, n + 1, (100_000,), generator=g, device=dev)
    e = (b + torch.randint(0, 257, (100_000,), generator=g, device=dev)).clamp(max=n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _check_ranges_on_device(ms, text, b, e, f"{ctx}: 10^5 random ranges")
    t_ranges = time.perf_counter() - t0
    # around every block cut (the ranks' text blocks) and at the end of the text
    edge = torch.arange(-300, 300, 7, device=dev)
    cb = (torch.tensor(cuts[1:-1], dtype=torch.int64, device=dev)[:, None] + edge).flatten().clamp(0, n)
    eb = torch.tensor([n - 1000, n - RATE - 1, n - 1, n, n], dtype=torch.int64, device=dev)
    ee = torch.tensor([n, n, n, n, n], dtype=torch.int64, device=dev)
    _check_ranges_on_device(ms, text, torch.cat([cb, eb]), torch.cat([(cb + 600).clamp(max=n), ee]),
                            f"{ctx}: ranges at the block cuts and the end")
    print(json.dumps({"case": case, "n": n, "ranks": world, "wide": bool(wide), "rate": RATE,
                      "isa_samples_s": round(t_isa, 4), "whole_text_s": round(t_whole, 4),
                      "ranges_1e5_checked_s": round(t_ranges, 4), "case_s": round(time.perf_counter() - t_case, 2),
                      "device_peak_bytes": torch.cuda.max_memory_allocated(dev), "computed_peak_bytes": need}),
          flush=True)
    del ms, text
    torch.cuda.empty_cache()
