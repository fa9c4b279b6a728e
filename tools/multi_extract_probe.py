"""Extract over the sliced index of the distributed build (MultiSliceIndex, csrc/extract.cu): inverse-SA samples,
whole-text extraction and 10^6 snippets of 64 symbols, each walk with the exact LF step across slices.

  c3_slices  the C3 text (ENG96 2*10^8 + '$') built by the single-GPU builder, its SA and BWT cut into 1, 2, 4 and 8
             slices, timed beside DeviceIndex's extract on the wavelet tree of the same index at the same rate: the
             cost of slicing.
  eng_2g     ENG96 2^31 + 2^26 + 1 symbols ('$' last) built by the distributed builder on 8 ranks emulated on one GPU.

Kernel time from CUDA events around the library calls (segment scan + walks), the median of `reps` after a warm-up,
with a 256 MiB buffer overwritten between repetitions (tools/extract_probe.py's Timer).  The device name and power
limit are read in the same run; every output is compared with the text in the same run.

    python tools/multi_extract_probe.py [--inputs c3_slices,eng_2g] [--reps 5] [--out DIR]
        -> DIR/r04_multi_extract_<input>.json
"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from extract_probe import E, Timer, _lib, device_info, extract_call, lf_steps  # noqa: E402
import torch  # noqa: E402
from hkcsa import dist_sa  # noqa: E402

RATES = (6, 32)


def multi_extract_call(ms, begin, end):
    """hkcsa_multi_extract into preallocated buffers: the timed region is the library call alone."""
    L = _lib.load()
    R = begin.numel()
    out_off = torch.zeros(R + 1, dtype=torch.int64, device="cuda")
    out_off[1:] = torch.cumsum(end - begin, 0)
    out = torch.empty(int(out_off[-1]), dtype=torch.uint8, device="cuda")
    nbytes = L.hkcsa_extract_scratch_bytes(R)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    isa = ms.isa_samples()

    def run():
        _lib.check(L.hkcsa_multi_extract(ms.desc.data_ptr(), ms.n, ms.rate, isa.data_ptr(), begin.data_ptr(),
                                         end.data_ptr(), out_off.data_ptr(), R, out.data_ptr(), scratch.data_ptr(),
                                         nbytes, torch.cuda.current_stream().cuda_stream))
    return run, out


def batches(n: int):
    gen = torch.Generator(device="cuda").manual_seed(7)
    b = torch.randint(0, n - 64 + 1, (1_000_000,), generator=gen, device="cuda", dtype=torch.int64)
    return {"whole_text": (torch.zeros(1, dtype=torch.int64, device="cuda"),
                           torch.full((1,), n, dtype=torch.int64, device="cuda")),
            "snippets_1000000x64": (b, b + 64)}


def time_extract(timer, make_call, text, bt, rate, label) -> dict:
    """Every batch through one extract call: time, symbols/s, LF steps/s; the output compared with the text."""
    n = text.numel()
    r = {}
    for name, (b, e) in bt.items():
        run, out = make_call(b, e)
        t = timer(run)
        want = text if name == "whole_text" else text[b[:, None] + torch.arange(64, device="cuda")].reshape(-1)
        assert torch.equal(out, want), f"{label} {name}: output differs from the text"
        del out, want
        syms, steps = int((e - b).sum()), lf_steps(b, e, rate, n)
        s = t["ms_median"] / 1e3
        t.update({"requests": int(b.numel()), "symbols": syms, "lf_steps": steps, "symbols_per_s": syms / s,
                  "lf_steps_per_s": steps / s, "output_checked": True})
        r[name] = t
        print(f"{label:28s} {name:20s} {t['ms_median']:9.3f} ms  {syms / s / 1e9:6.2f} G sym/s", flush=True)
    return r


def time_isa(timer, ms, label) -> dict:
    def isa_run():
        ms._isa = None
        ms.isa_samples()
    t = timer(isa_run)
    t["samples"] = int(ms.isa_samples().numel() - 1)
    print(f"{label:28s} {'isa_samples':20s} {t['ms_median']:9.3f} ms", flush=True)
    return t


def probe_c3_slices(reps: int) -> dict:
    text = torch.cat([E.gen_text(E.ENG96, 42, 200_000_000), torch.tensor([0x24], dtype=torch.uint8, device="cuda")])
    n = text.numel()
    timer = Timer(reps)
    res = {"input": "c3_slices", "n": n, "reps": reps, "l2_flush_bytes": 256 << 20, **device_info(), "rates": {}}
    bt = batches(n)
    for rate in RATES:
        idx = E.DeviceIndex(text, sa_sample_rate=rate)
        r = {"wavelet_levels": idx.wt.levels, "sigma": idx.wt.sigma}
        # the reference: DeviceIndex's extract on the wavelet tree of the same index
        label = f"rate {rate} single index"

        def isa_run():
            idx._isa = None
            idx.isa_samples()
        r["single_index"] = {"isa_samples": timer(isa_run),
                             **time_extract(timer, lambda b, e: extract_call(idx, b, e, None), text, bt, rate, label)}
        sa, bwt = idx.sa, idx.bwt
        for parts in (1, 2, 4, 8):
            cuts = [n * k // parts for k in range(parts + 1)]
            ms = dist_sa.MultiSliceIndex(n, [{"bwt": bwt[a:b], "sa": sa[a:b]} for a, b in zip(cuts[:-1], cuts[1:])],
                                         sa_sample_rate=rate)
            label = f"rate {rate} {parts} slice(s)"
            want = idx.isa_samples().to(torch.int64)
            assert torch.equal(ms.isa_samples(), want), f"{label}: inverse samples differ from the single index's"
            r[f"slices_{parts}"] = {"isa_samples": time_isa(timer, ms, label),
                                    **time_extract(timer, lambda b, e: multi_extract_call(ms, b, e), text, bt, rate,
                                                   label)}
            del ms
            torch.cuda.empty_cache()
        res["rates"][str(rate)] = r
        del idx, sa, bwt
        torch.cuda.empty_cache()
    return res


def probe_eng_2g(reps: int) -> dict:
    n = (1 << 31) + (1 << 26) + 1
    text = torch.cat([E.gen_text(E.ENG96, 42, n - 1), torch.tensor([0x24], dtype=torch.uint8, device="cuda")])
    world = 8
    cuts = [n * k // world for k in range(world + 1)]
    t0 = time.perf_counter()
    slices = dist_sa.emulate_distributed_suffix_array([text[cuts[k]:cuts[k + 1]] for k in range(world)])
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    ms = dist_sa.MultiSliceIndex(n, [{"bwt": sl.bwt, "sa": sl.sa} for sl in slices], sa_sample_rate=32)
    del slices
    torch.cuda.empty_cache()
    timer = Timer(reps)
    res = {"input": "eng_2g", "n": n, "ranks": world, "rate": 32, "reps": reps, "l2_flush_bytes": 256 << 20,
           **device_info(), "emulated_build_s": round(t_build, 2), "slice_sizes": [int(s) for s in
                                                                                    torch.tensor(ms.starts).diff()]}
    res["isa_samples"] = time_isa(timer, ms, "eng_2g 8 ranks")
    res.update(time_extract(timer, lambda b, e: multi_extract_call(ms, b, e), text, batches(n), 32, "eng_2g 8 ranks"))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--inputs", default="c3_slices,eng_2g")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for r04_multi_extract_<input>.json (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_extract_probe needs a CUDA device")
    for name in args.inputs.split(","):
        res = {"c3_slices": probe_c3_slices, "eng_2g": probe_eng_2g}[name](args.reps)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r04_multi_extract_{name}.json"), "w") as f:
                json.dump(res, f, indent=1)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
