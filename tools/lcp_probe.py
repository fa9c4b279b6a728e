"""LCP (csrc/lcp.cu) timings: hkcsa_lcp_build (LCP only, PLCP only), the steps of DeviceIndex.build_lcp_bits (PLCP,
hkcsa_plcp_bits, the bit-vector build of each piece) and lcp_rows of 10^6 random rows (sampled-SA locate at rate 32
and full-SA locate), beside the suffix-array build of the same text in the same run.  Workloads: C2 (DNA 10^8 + '$'),
C3 (ENG96 2*10^8 + '$'), DNA at HKCSA_MAX_N, Fibonacci at 2^27, "mississippi$" repeated to 10^8 symbols.  CUDA events
around the library calls after a warm-up call, with a 256 MiB buffer overwritten between repetitions so that no
repetition finds the previous one's lines in L2 (every input is larger than L2).  Every LCP array is compared with
the PLCP array through the suffix array, and lcp_rows with the LCP array, in the same run.

    python tools/lcp_probe.py [--workloads c2,c3,dna_max,fib27,mississippi] [--reps 5] [--out DIR]
        -> DIR/r06_lcp_<workload>.json
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "high-order-entropy-compressed-suffix-array_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from extract_probe import Timer, device_info  # noqa: E402
from hkcsa import _lib, engine as E  # noqa: E402


def _fib(n: int) -> bytes:
    a, b = b"a", b"ab"
    while len(b) < n:
        a, b = b, b + a
    return b[:n]


def _text(name: str) -> torch.Tensor:
    dollar = torch.tensor([0x24], dtype=torch.uint8, device="cuda")
    if name == "c2":
        return torch.cat([E.gen_text(E.DNA4, 43, 100_000_000), dollar])
    if name == "c3":
        return torch.cat([E.gen_text(E.ENG96, 42, 200_000_000), dollar])
    if name == "dna_max":
        return torch.cat([E.gen_text(E.DNA4, 43, _lib.MAX_N - 1), dollar])
    if name == "fib27":
        return E.to_device_u8(_fib((1 << 27) - 1) + b"$")
    if name == "mississippi":
        return E.to_device_u8((b"mississippi$" * (100_000_000 // 12 + 1))[:100_000_000])
    raise ValueError(name)


def probe(name: str, reps: int) -> dict:
    L = _lib.load()
    text = _text(name)
    n = text.numel()
    timer = Timer(reps)
    st = torch.cuda.current_stream().cuda_stream
    res = {"workload": name, "n": n, "reps": reps, "l2_flush_bytes": 256 << 20, **device_info()}
    # ---- suffix array (the same call DeviceIndex's build starts with), then the LCP build on it
    sa = torch.empty(n, dtype=torch.int32, device="cuda")
    sa_bytes = L.hkcsa_sa_scratch_bytes(n)
    sa_scratch = torch.empty(sa_bytes, dtype=torch.uint8, device="cuda")
    res["sa_build"] = timer(lambda: _lib.check(L.hkcsa_sa_build(text.data_ptr(), n, sa.data_ptr(), sa_scratch.data_ptr(),
                                                                  sa_bytes, st, None)))
    del sa_scratch
    torch.cuda.empty_cache()
    lcp = torch.empty(n, dtype=torch.int32, device="cuda")
    plcp = torch.empty(n, dtype=torch.int32, device="cuda")
    nbytes = L.hkcsa_lcp_scratch_bytes(n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    res["lcp_scratch_bytes_per_symbol"] = nbytes / n

    def build(out_lcp, out_plcp, stats=None):
        return lambda: _lib.check(L.hkcsa_lcp_build(text.data_ptr(), n, sa.data_ptr(), out_lcp, out_plcp,
                                                    scratch.data_ptr(), nbytes, stats, st))
    res["lcp_build_lcp_only"] = timer(build(lcp.data_ptr(), None))
    res["lcp_build_plcp_only"] = timer(build(None, plcp.data_ptr()))
    h = (C.c_uint64 * 2)()
    build(None, plcp.data_ptr(), h)()
    res["irreducible_positions"], res["irreducible_sum"] = int(h[0]), int(h[1])
    res["irreducible_sum_over_n"] = int(h[1]) / n
    res["irreducible_sum_bound_2nlog2n"] = 2 * n * float(np.log2(n))
    rounds = 0
    while (32 << rounds) < n:
        rounds += 1
    res["rounds_launched"] = rounds
    assert torch.equal(lcp, plcp[sa.long()]), f"{name}: LCP != PLCP[SA]"
    for k in ("sa_build", "lcp_build_lcp_only", "lcp_build_plcp_only"):
        res[k]["ns_per_symbol"] = res[k]["ms_median"] * 1e6 / n
    # ---- the steps of build_lcp_bits and lcp_rows, on an index with a sampled SA
    del scratch, lcp
    torch.cuda.empty_cache()
    idx = E.DeviceIndex(text, sa_sample_rate=32)
    bits = torch.empty(2 * n, dtype=torch.uint8, device="cuda")
    res["plcp_bits"] = timer(lambda: _lib.check(L.hkcsa_plcp_bits(plcp.data_ptr(), n, bits.data_ptr(), st)))
    cut = _lib.MAX_N
    res["bitvec_build_pieces"] = [timer(lambda a=a: E.DeviceBitVector(bits[a:a + cut])) for a in range(0, 2 * n, cut)]
    del bits
    idx.build_lcp_bits()
    res["lcp_bits_per_symbol"] = idx._lcp_bits_held() / n
    want = idx.lcp()
    rows = torch.randint(0, n, (1_000_000,), device="cuda", dtype=torch.int32,
                         generator=torch.Generator(device="cuda").manual_seed(9))
    for mode, samples in (("lcp_rows_sampled_sa_rate32", True), ("lcp_rows_full_sa", False)):
        out = {}
        res[mode] = timer(lambda s=samples: out.__setitem__("v", idx.lcp_rows(rows, use_samples=s)))
        assert torch.equal(out["v"], want[rows.long()]), f"{name}: {mode} differs from the LCP array"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3,dna_max,fib27,mississippi")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    for w in a.workloads.split(","):
        r = probe(w, a.reps)
        with open(os.path.join(a.out, f"r06_lcp_{w}.json"), "w") as f:
            json.dump(r, f, indent=1)
        print(json.dumps({k: (v["ms_median"] if isinstance(v, dict) and "ms_median" in v else v)
                          for k, v in r.items() if k != "bitvec_build_pieces"}), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
