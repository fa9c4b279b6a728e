"""Count and locate over the sliced index of the distributed build (MultiSliceIndex; both kernels in
csrc/fm_search.cu): the C3 text (ENG96 2*10^8 + '$') built by the single-GPU builder at sampling rate 32, its SA and
BWT cut into 1, 2, 4 and 8 slices.

  count   MultiSliceIndex.count_batch of 10^6 seeded patterns of length 8-64 (half with one substitution)
  locate  MultiSliceIndex.locate_rows of 10^6 random rows: LF walks across the slices to a marked row

Time from CUDA events around the calls, the median of `reps` after a warm-up, with a 256 MiB buffer overwritten
between repetitions (tools/extract_probe.py's Timer).  The device name and power limit are read in the same run; the
ranges and positions of every slicing are compared with the single index's in the same run.

    python tools/multi_query_probe.py [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from extract_probe import E, Timer, device_info  # noqa: E402
import torch  # noqa: E402
from hkcsa import dist_sa  # noqa: E402

P = 1_000_000
ROWS = 1_000_000
RATE = 32


def probe(reps: int) -> dict:
    text = torch.cat([E.gen_text(E.ENG96, 42, 200_000_000), torch.tensor([0x24], dtype=torch.uint8, device="cuda")])
    n = text.numel()
    idx = E.DeviceIndex(text, sa_sample_rate=RATE)
    alpha = torch.unique(text[: 1 << 22])
    alpha = alpha[alpha != 0x24]
    pats, off = E.gen_patterns(44, P, text[: n - 1], alpha)
    lo, hi = idx.count_batch(pats, off)
    gen = torch.Generator(device="cuda").manual_seed(7)
    rows = torch.randint(0, n, (ROWS,), generator=gen, device="cuda", dtype=torch.int64)
    want_pos = idx.sa[rows].to(torch.int64) & 0xFFFFFFFF
    sa, bwt = idx.sa, idx.bwt
    timer = Timer(reps)
    res = {"input": "c3_slices", "n": n, "rate": RATE, "count_patterns": P, "locate_rows": ROWS, "reps": reps,
           "l2_flush_bytes": 256 << 20, **device_info(), "slices": {}}
    for parts in (1, 2, 4, 8):
        cuts = [n * k // parts for k in range(parts + 1)]
        ms = dist_sa.MultiSliceIndex(n, [{"bwt": bwt[a:b], "sa": sa[a:b]} for a, b in zip(cuts[:-1], cuts[1:])],
                                     sa_sample_rate=RATE)
        mlo, mhi = ms.count_batch(pats, off)
        assert torch.equal(mlo, lo) and torch.equal(mhi, hi), f"{parts} slice(s): ranges differ from the single index's"
        assert torch.equal(ms.locate_rows(rows), want_pos), f"{parts} slice(s): positions differ from the SA"
        tc = timer(lambda: ms.count_batch(pats, off))
        tl = timer(lambda: ms.locate_rows(rows))
        tc["patterns_per_s"] = P / (tc["ms_median"] / 1e3)
        tl["rows_per_s"] = ROWS / (tl["ms_median"] / 1e3)
        res["slices"][str(parts)] = {"count": tc, "locate": tl, "checked": True}
        print(f"{parts} slice(s)  count {tc['ms_median']:8.3f} ms {tc['patterns_per_s'] / 1e9:6.3f} G patterns/s   "
              f"locate {tl['ms_median']:8.3f} ms {tl['rows_per_s'] / 1e9:6.3f} G rows/s", flush=True)
        del ms
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="JSON file for the result (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_query_probe needs a CUDA device")
    res = probe(args.reps)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
