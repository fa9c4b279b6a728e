"""Extract (csrc/extract.cu) on the C2 (DNA 10^8 + '$') and C3 (ENG96 2*10^8 + '$') workloads at sampling rates 6 and
32: inverse-SA samples, whole-text extraction and random snippets, each LF step on the wavelet tree and on the sampled
Occ table (layout 1).  Kernel time from CUDA events around the library calls (segment scan + walks), after a warm-up,
with a 256 MiB buffer overwritten between repetitions so that no repetition finds the previous one's lines in L2.
Every output is compared with the generated text in the same run.

    python tools/extract_probe.py [--corpora c2,c3] [--reps 5] [--out DIR]    -> DIR/r03_extract_<corpus>.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "high-order-entropy-compressed-suffix-array_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from hkcsa import _lib, engine as E  # noqa: E402

CORPORA = {"c2": (E.DNA4, 43, 100_000_000), "c3": (E.ENG96, 42, 200_000_000)}
SECTOR_CEILING = 40e9          # random 32-byte requests/s of one B200 (tools/probes/sector_probe.cu)


def device_info() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:                       # read-only query
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")[:2]]
    except Exception as e:     # noqa: BLE001
        info["power_limit"] = f"unavailable ({e})"
    return info


class Timer:
    def __init__(self, reps):
        self.reps = reps
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self, fn) -> dict:
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(self.reps):
            self.flush.fill_(len(ms) & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return {"ms_median": float(np.median(ms)), "ms_min": float(min(ms)), "ms_all": [round(x, 4) for x in ms]}


def extract_call(idx, begin, end, occ):
    """hkcsa_extract into preallocated buffers: the timed region is the library call alone."""
    L = _lib.load()
    R = begin.numel()
    out_off = torch.zeros(R + 1, dtype=torch.int64, device="cuda")
    out_off[1:] = torch.cumsum(end - begin, 0)
    out = torch.empty(int(out_off[-1]), dtype=torch.uint8, device="cuda")
    nbytes = L.hkcsa_extract_scratch_bytes(R)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    isa = idx.isa_samples()
    plan, blob = occ if occ is not None else (None, None)

    def run():
        _lib.check(L.hkcsa_extract(idx.wt.blob.data_ptr(), C.byref(idx.wt.plan), blob.data_ptr() if blob is not None else None,
                                   C.byref(plan) if plan is not None else None, isa.data_ptr(), int(idx.ssa.plan.rate),
                                   begin.data_ptr(), end.data_ptr(), out_off.data_ptr(), R, out.data_ptr(),
                                   scratch.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream))
    return run, out


def lf_steps(begin: torch.Tensor, end: torch.Tensor, rate: int, n: int) -> int:
    """LF steps of a batch: every symbol emitted plus the steps a walk makes past `end` to reach it from the next
    sample (the last segment of each request starts at min(ceil(end / rate) * rate, n))."""
    start = torch.clamp(torch.div(end + rate - 1, rate, rounding_mode="floor") * rate, max=n)
    return int((end - begin).sum()) + int((start - end).sum())


def probe(corpus: str, reps: int) -> dict:
    kind, seed, n0 = CORPORA[corpus]
    text = torch.cat([E.gen_text(kind, seed, n0), torch.tensor([0x24], dtype=torch.uint8, device="cuda")])
    n = text.numel()
    timer = Timer(reps)
    res = {"corpus": corpus, "n": n, "reps": reps, "l2_flush_bytes": 256 << 20, **device_info(), "rates": {}}
    gen = torch.Generator(device="cuda").manual_seed(7)
    batches = {"whole_text": (torch.zeros(1, dtype=torch.int64, device="cuda"),
                              torch.full((1,), n, dtype=torch.int64, device="cuda"))}
    for R, m in ((1_000_000, 64), (100_000, 4096)):
        b = torch.randint(0, n - m + 1, (R,), generator=gen, device="cuda", dtype=torch.int64)
        batches[f"snippets_{R}x{m}"] = (b, b + m)
    for rate in (6, 32):
        idx = E.DeviceIndex(text, sa_sample_rate=rate, keep_sa=False)
        levels = idx.wt.levels
        r = {"wavelet_levels": levels, "sigma": idx.wt.sigma}
        S = int(idx.ssa.plan.n_samples)

        def isa_run():
            idx._isa = None
            idx.isa_samples()
        r["isa_samples"] = timer(isa_run)
        r["isa_samples"]["samples"] = S
        occ = idx.build_occ_table(5, layout=1)
        idx.bwt = None
        for name, (b, e) in batches.items():
            steps = lf_steps(b, e, rate, n)
            syms = int((e - b).sum())
            want = text if name == "whole_text" else text[b[:, None] + torch.arange(int(e[0] - b[0]), device="cuda")].reshape(-1)
            for lf, occ_arg, per_step in (("wavelet_tree", None, levels), ("occ_layout1", occ, 2)):
                run, out = extract_call(idx, b, e, occ_arg)
                t = timer(run)
                assert torch.equal(out, want), f"{corpus} rate {rate} {name} {lf}: output differs from the text"
                s = t["ms_median"] / 1e3
                t.update({"requests": int(b.numel()), "symbols": syms, "lf_steps": steps,
                          "symbols_per_s": syms / s, "lf_steps_per_s": steps / s,
                          "memory_requests_per_lf_step": per_step,
                          "memory_requests_per_s": steps * per_step / s,
                          "share_of_sector_ceiling": steps * per_step / s / SECTOR_CEILING, "output_checked": True})
                r[f"{name}/{lf}"] = t
                print(f"{corpus} rate {rate:2d} {name:24s} {lf:13s} {t['ms_median']:9.3f} ms  "
                      f"{syms / s / 1e9:6.2f} G sym/s  {steps * per_step / s / 1e9:6.2f} G req/s", flush=True)
            del want
        print(f"{corpus} rate {rate:2d} isa_samples {r['isa_samples']['ms_median']:.3f} ms ({S} samples)", flush=True)
        res["rates"][str(rate)] = r
        del idx, occ
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--corpora", default="c2,c3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for r03_extract_<corpus>.json (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("extract_probe needs a CUDA device")
    for corpus in args.corpora.split(","):
        res = probe(corpus, args.reps)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r03_extract_{corpus}.json"), "w") as f:
                json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
