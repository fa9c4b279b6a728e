"""The distributed build (hkcsa.dist_sa) and the sliced index it leaves behind, at the sizes it exists for, checked
against the exact torch references of tests/device_reference.py on the device.

The ranks are emulated on one GPU by emulate_distributed_suffix_array: the same per-rank program, pack-and-exchange
kernel, sort, group round, extension rounds and rank doubling that torchrun runs, with the peers' buffers local.
  eng_2g        2^31 + 2^26 + 1 symbols on 8 ranks, 32-bit ids: ids >= 2^31 stored in int32 tensors, cut points from
                sampled histograms and exact owner counts (every block >= 2^24), slices of ~2^28;
  dna_wide      2^30 + 2^20 + 1 symbols on 5 uneven ranks, 64-bit ids forced: receive arrays of 64-bit ids with key
                extension bits and the BWT symbol in the top byte, gather_ids64, the wide group round;
  mississippi   "mississippi$" * floor(2^28 / 12) on 8 ranks: rank doubling over the emulated peers' ISA blocks, and a
                last symbol that recurs;
  block_repeat  one 1 MiB English-like block x 256, then '$', on 8 ranks: doubling plus the search that ranks suffixes
                which became unique before it (dsa_remote_rank).
Each case checks the slices (offsets, the suffix array, the BWT) and a MultiSliceIndex over them at sampling rate 32:
count against suffix-array ranges, locate of single rows and of whole pattern ranges.

One build per case, freed before the next.  A case skips only when the device reports less free memory than its
computed peak (the number is in the reason).  HKCSA_ENVELOPE_SCALE = 2^j (default 1) divides every n, for a quick
rehearsal."""
import json
import os
import time

import pytest
import torch

import device_reference as R
from test_gpu_envelope import DOLLAR, GB, SCALE, _csr, _join, _no_inner_sentinel, _subset

pytestmark = pytest.mark.gpu

RATE = 32


def _dollar(dev):
    return torch.tensor([DOLLAR], dtype=torch.uint8, device=dev)


def _even(world):
    return [r / world for r in range(world + 1)]


# name -> (n, make(E, n, dev) -> uint8 text, block fractions, wide, text is repetitive, largest slice / mean slice)
def _cases():
    k = ((1 << 28) // SCALE) // 12
    blk = (1 << 20) // SCALE
    return {
        "eng_2g": (((1 << 31) + (1 << 26)) // SCALE + 1,
                   lambda E, n, d: torch.cat([E.gen_text(E.ENG96, 42, n - 1), _dollar(d)]), _even(8), None, False, 1.05),
        "dna_wide": (((1 << 30) + (1 << 20)) // SCALE + 1,
                     lambda E, n, d: torch.cat([E.gen_text(E.DNA4, 43, n - 1), _dollar(d)]),
                     [0, 0.13, 0.35, 0.52, 0.8, 1], True, False, 1.05),
        "mississippi": (12 * k, lambda E, n, d: torch.tensor(list(b"mississippi$"), dtype=torch.uint8,
                                                             device=d).repeat(k), _even(8), None, True, 1.4),
        "block_repeat": (256 * blk + 1, lambda E, n, d: torch.cat([E.gen_text(E.ENG96, 44, blk).repeat(256), _dollar(d)]),
                         _even(8), None, True, 1.05),
    }


CASES = _cases()


@pytest.fixture(scope="module")
def E(cuda):
    from hkcsa import engine
    return engine


def _peak_bytes(n, wide, skew):
    """While the emulated ranks hold their workspaces, per symbol: the receive arrays (8 B keys + two 4 B value
    arrays, + 8 B ids when wide) and the carve_dsa scratch (25.3 B), every rank's sized by the largest slice (`skew`
    x the mean: 12 buckets over 8 ranks on "mississippi$"); the ISA blocks (4 or 8 B); the slices (ids + BWT); the
    test's text and the replicated one.  Measured with torch.cuda.max_memory_allocated (DESIGN section 5), the test's
    text included: 52.4 B/symbol with 32-bit ids and even slices, 68.4 with 64-bit ids, 66.6 on "mississippi$"; the
    formula gives 54.4 / 70.8 / 68.8 there.
    After the build the checks hold the int64 SA and ISA, the slices, the text and the sliced index: ~30 B/symbol."""
    per = (16 + (8 if wide else 0) + 25.3) * skew + (8 if wide else 4) + (9 if wide else 5) + 2
    return int(n * per) + 4 * GB


@pytest.mark.parametrize("case", list(CASES))
def test_distributed_build_at_scale(E, case):
    from hkcsa import dist_sa
    n, make, frac, wide, repetitive, skew = CASES[case]
    dev = torch.device("cuda", 0)
    torch.cuda.empty_cache()
    need = _peak_bytes(n, bool(wide), skew)
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need:
        pytest.skip(f"{case}: needs {need / GB:.1f} GiB of device memory, {free / GB:.1f} GiB free")
    text = make(E, n, dev)
    assert text.numel() == n and int(text[-1]) == DOLLAR
    cuts = [int(n * f) for f in frac]
    world = len(cuts) - 1
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    t0 = time.perf_counter()
    slices = dist_sa.emulate_distributed_suffix_array([text[cuts[r]:cuts[r + 1]] for r in range(world)], wide=wide)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    build_peak = torch.cuda.max_memory_allocated(dev) - base
    ext = max(sl.ext_rounds for sl in slices)
    dbl = max(sl.dbl_rounds for sl in slices)
    ctx = f"{case}: n={n}, ranks={world}, ext_rounds={ext}, dbl_rounds={dbl}"

    # ---- 1. the slices: contiguous in rank order, the suffix array and the BWT
    off = 0
    for sl in slices:
        assert sl.offset == off and sl.n == n, ctx
        assert sl.sa.dtype == (torch.int64 if wide else torch.int32) and sl.bwt.numel() == sl.sa.numel(), ctx
        off += sl.sa.numel()
    assert off == n, ctx
    if repetitive:
        assert dbl >= 1, ctx
    sa = torch.cat([sl.sa_int64() for sl in slices])
    if case == "eng_2g":           # ids past 2^31 are stored as uint32 bit patterns in the int32 slices
        assert any(bool((sl.sa < 0).any()) for sl in slices) == (n > (1 << 31)), ctx
    try:
        isa = R.check_suffix_array(text, sa)
    except AssertionError as err:
        raise AssertionError(f"{ctx}: {err}") from None
    assert torch.equal(torch.cat([sl.bwt for sl in slices]), R.bwt_of(text, sa)), f"{ctx}: BWT"
    row0 = int(isa[0])
    del isa

    # ---- 2. the sliced index at rate 32
    ms = dist_sa.MultiSliceIndex(n, [{"bwt": sl.bwt, "sa": sl.sa} for sl in slices], sa_sample_rate=RATE)
    for sl in slices:
        sl.text = None                     # the replicated text: the test's own copy serves the checks
    assert ms.row0 == row0, ctx
    starts = torch.tensor(ms.starts, dtype=torch.int64, device=dev)
    g = torch.Generator(device=dev).manual_seed(n)
    # count: windows of length 1..64 starting at the suffixes on both sides of every slice boundary and at the text
    # positions on both sides of every block boundary, random substrings, misses and the empty pattern
    edge = torch.arange(-16, 16, device=dev)
    brows = (starts[1:-1, None] + edge).flatten().clamp(0, n - 1)
    bpos = (torch.tensor(cuts[1:-1], dtype=torch.int64, device=dev)[:, None] + edge).flatten().clamp(0, n - 1)
    wstart = torch.cat([sa[brows], bpos])
    wlen = torch.minimum(torch.randint(1, 65, (wstart.numel(),), generator=g, device=dev), n - wstart)
    present = torch.bincount(text[: min(n, 1 << 24)].long(), minlength=256).nonzero().flatten().to(torch.uint8)
    npat = (1 << 16) - wstart.numel() - 257
    pats, poff = E.gen_patterns(n % 1000, npat, text[: n - 1], present[present != DOLLAR], 1, 64)
    absent = (torch.randint(0, 256, (256 * 12,), generator=g, device=dev).to(torch.uint8),
              torch.arange(0, 257 * 12, 12, device=dev))
    empty = (torch.zeros(0, dtype=torch.uint8, device=dev), torch.zeros(2, dtype=torch.int64, device=dev))
    pats, poff = _no_inner_sentinel(*_join(_csr(text, wstart, wlen), (pats, poff), absent, empty))
    lo, hi = R.sa_range(text, sa, pats, poff)
    got = ms.count_batch(pats, poff)
    assert torch.equal(got[0], lo) and torch.equal(got[1], hi), f"{ctx}: count of {lo.numel()} patterns"
    # locate of single rows: random, every slice boundary +- 1, the row of suffix 0 +- 1
    qrows = torch.cat([torch.randint(0, n, (1 << 20,), generator=g, device=dev),
                       (starts[1:-1, None] + torch.arange(-1, 2, device=dev)).flatten(),
                       torch.arange(row0 - 1, row0 + 2, device=dev)]).clamp(0, n - 1)
    assert torch.equal(ms.locate_rows(qrows), sa[qrows]), f"{ctx}: locate_rows"
    # locate of whole ranges: every pattern with at most 1024 occurrences and the present one with the fewest
    cnt = torch.where(lo >= 0, hi - lo + 1, torch.zeros_like(lo))
    few = cnt <= 1024
    few[torch.where(cnt > 0, cnt, torch.full_like(cnt, n + 1)).argmin()] = True
    lp, lo_ = _subset(pats, poff, few)
    o, p = ms.locate_batch(lp, lo_)
    located = f"{ctx}: locate_batch of {int(few.sum())} patterns, {int(o[-1])} positions"
    assert int(o[-1]) > 0 and torch.equal(o[1:] - o[:-1], cnt[few]), located
    first = torch.repeat_interleave(lo[few], cnt[few])
    first = first + torch.arange(first.numel(), device=dev) - torch.repeat_interleave(o[:-1], cnt[few])
    assert torch.equal(p, sa[first]), located
    print(json.dumps({"case": case, "n": n, "ranks": world, "wide": bool(wide), "ext_rounds": ext, "dbl_rounds": dbl,
                      "build_s": round(t_build, 2), "build_peak_bytes": build_peak,
                      "build_peak_bytes_per_symbol": round(build_peak / n, 2),
                      "computed_peak_bytes": need, "device_peak_bytes": torch.cuda.max_memory_allocated(dev),
                      "slice_sizes": [int(sl.sa.numel()) for sl in slices],
                      "patterns": int(lo.numel()), "located": int(o[-1])}), flush=True)
    del ms, slices, sa, text, first, p, o
    torch.cuda.empty_cache()
