#!/usr/bin/env python
"""bench.py -- index build MB/s (SA + BWT + wavelet tree) and batched count / locate
throughput of the B200 hot path, with the reference's CPU path timed beside it.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # reference arm (CPU oracle port)
    python bench.py ... --dump-outputs DIR                   # + the last timed build's outputs as DIR/*.npy

One step = one full index build of the workload text: byte histogram -> K1 suffix
array -> K2 BWT -> K3 wavelet tree with rank/select directories and C[] -> sampled
SA.  Default workload = BASELINE.json configs[1]: 100 MB synthetic DNA (sigma 4,
order-5 Markov, seed 43) + '$'.  N > 1 (torchrun): N independent replicas, one per
GPU ("replicas only", DESIGN.md), value = N * text bytes / max-over-ranks time;
the count queries that follow are sharded over the ranks (index replicated).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "high-order-entropy-compressed-suffix-array_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {
    # name: (generator kind, seed, text bytes, description)
    "c1": (0, 42, 1 << 20, "1 MiB ENG96 order-3 Markov text + '$' (BASELINE configs[0])"),
    "c2": (1, 43, 100_000_000, "100 MB DNA4 order-5 Markov text + '$' (BASELINE configs[1])"),
    "c3": (0, 42, 200_000_000, "200 MB ENG96 order-3 Markov text + '$' (BASELINE configs[2])"),
}
METRIC = "index build MB/s (SA+BWT+WT)"
TOP_KERNEL_CLASS = "onesweep_u64"     # the dominant kernel (share of the step checked in profiles/): timed live
SA_SAMPLE_RATE = 32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--size", type=int, default=0, help="override the text size in bytes (debug)")
    ap.add_argument("--patterns", type=int, default=10_000_000, help="count queries after the build (C4 shape)")
    ap.add_argument("--cpu-sample", type=int, default=32_000_000, help="bytes of the workload the CPU baseline builds")
    ap.add_argument("--ref-sample", type=int, default=0, help="--impl reference: build only a prefix (0 = whole text)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dist-build", action="store_true", help="N > 1: skip the distributed-build record")
    ap.add_argument("--dist-bytes-per-rank", type=int, default=1_000_000_000)
    ap.add_argument("--no-c3", action="store_true", help="skip the C3 / C4 records (200 MB ENG96 text)")
    ap.add_argument("--no-queries", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed build computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (NVML, every 20 ms; falls back to
    nvidia-smi polling)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        nv = self._nvml
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                          ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                          ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
        if out.returncode == 0 and out.stdout.strip():
            r = [x.strip() for x in out.stdout.strip().split(",")]
            self.sm.append(float(r[0]))
            self.sm_max = float(r[1])
            for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if r[2 + i].lower() == "active":
                    self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.02 if self._nvml is not None else 0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self._nvml is not None else "nvidia-smi"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ------------------------------------------------------------------ reference arm / CPU baseline
def cpu_build_sample(kind, seed, nbytes):
    """The oracle port of the reference's build path on a bounded sample of the workload:
    build_suffix_array(text+'$') -> bwt_transform -> WaveletTree(bwt) spine + rank_support + C[]."""
    from oracle import oracle as O
    text = O.gen_text(kind, seed, nbytes).tobytes() + b"$"
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    sa = O.build_suffix_array(text, threads=threads)
    bwt = O.bwt_transform(text, sa)
    O.build_count(text)
    _, levels = O.wt_spine(bwt)
    for bits in levels:
        O.rank_support(bits)
    dt = time.perf_counter() - t0
    return dt, threads, len(text)


def run_reference(args):
    kind, seed, nbytes, desc = WORKLOADS[args.workload]
    if args.size:
        nbytes = args.size
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the whole workload text every step (the same config as the GPU arm): suffix sorting is super-linear, a
    # prefix would flatter the CPU
    sample = nbytes if not args.ref_sample else min(nbytes, args.ref_sample)
    times = []
    threads = 1
    for i in range(args.warmup + args.steps):
        dt, threads, n = cpu_build_sample(kind, seed, sample)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / 1e6 / (ms / 1e3)
    sample_desc = (f"the whole workload text ({sample} bytes + '$')" if sample == nbytes else
                   f"first {sample} bytes of the workload text (+'$')") + f", oracle port of SA+BWT+WT, {threads} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32/u64 integer", "data": "synthetic",
        "config": {"workload": desc, "text_bytes": nbytes, "index_symbols": nbytes + 1, "cpu_sample_bytes": sample,
                   "same_config_as_gpu_arm": sample == nbytes},
        "cpu_baseline": {"value": value, "unit": "MB/s", "cores": threads, "kind": "port", "sample": sample_desc},
        "e2e": {"value": value, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ distributed build record (N > 1)
NVLINK_GBS = 900.0       # per direction per GPU (NVLink 5)


def _suffix_order_violations(text, ids_a, ids_b, width=96):
    """Pairs (a, b) of suffix ids that must satisfy suffix(a) < suffix(b): compares the first `width` symbols on the
    device (the end of the text is smallest); returns (violations, undecided within `width`)."""
    import torch
    n = text.numel()
    ar = torch.arange(width, device=text.device, dtype=torch.int64)
    pa, pb = ids_a[:, None] + ar, ids_b[:, None] + ar
    A = torch.where(pa < n, text[pa.clamp(max=n - 1)].to(torch.int16), torch.full_like(pa, -1, dtype=torch.int16))
    B = torch.where(pb < n, text[pb.clamp(max=n - 1)].to(torch.int16), torch.full_like(pb, -1, dtype=torch.int16))
    diff = A != B
    has = diff.any(1)
    first = diff.to(torch.int8).argmax(1)
    a1 = A.gather(1, first[:, None])[:, 0]
    b1 = B.gather(1, first[:, None])[:, 0]
    bad = has & (a1 > b1)
    return int(bad.sum().item()), int((~has).sum().item())


def run_dist_build(args, world, rank, dev, barrier, max_over_ranks, sum_over_ranks, peak):
    import torch
    import torch.distributed as dist
    from hkcsa import dist_sa, engine as E, _lib
    L = _lib.load()
    out = {}

    def make_blocks(kind, seed, n_total):
        full = torch.empty(n_total, dtype=torch.uint8, device=dev)
        E.check(L.hkcsa_gen_text(kind, seed, n_total - 1, full.data_ptr(), torch.cuda.current_stream().cuda_stream))
        full[n_total - 1] = 0x24
        per = n_total // world
        blk = full[rank * per:(rank + 1) * per if rank < world - 1 else n_total].clone()
        return full, blk

    try:
        # ---- parity leg: N x 100 MB (<= HKCSA_MAX_N), the same text built on ONE GPU in the same run: this rank's
        #      slice must equal its range of the single-GPU suffix array and BWT bit for bit
        n_par = min(100_000_000 * world, 900_000_000) // world * world
        full, blk = make_blocks(0, 42, n_par)
        sl = dist_sa.distributed_suffix_array(blk)
        ref_sa = E.suffix_array(full)
        ref_bwt = E.bwt(full, ref_sa)
        lo_, hi_ = sl.offset, sl.offset + sl.sa.numel()
        ok = bool(torch.equal(sl.sa, ref_sa[lo_:hi_])) and bool(torch.equal(sl.bwt, ref_bwt[lo_:hi_]))
        covered = sum_over_ranks(float(sl.sa.numel()))
        out["parity"] = {"text_bytes": n_par, "workload": "ENG96 + '$'",
                         "slices_equal_single_gpu_sa_and_bwt": sum_over_ranks(1.0 if ok else 0.0) == world,
                         "slices_cover_n": covered == n_par}
        assert out["parity"]["slices_equal_single_gpu_sa_and_bwt"] and out["parity"]["slices_cover_n"], "distributed build differs"
        # the reference benchmark's own workload (tests/benchmark.py:110), scaled: LCPs of megabytes -> rank doubling
        reps_ = 1_000_000
        miss = torch.from_numpy(np.frombuffer(b"mississippi$" * reps_, dtype=np.uint8).copy()).to(dev)
        per = miss.numel() // world
        mblk = miss[rank * per:(rank + 1) * per if rank < world - 1 else miss.numel()].clone()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        slm = dist_sa.distributed_suffix_array(mblk)
        torch.cuda.synchronize()
        t_rep = max_over_ranks(time.perf_counter() - t0)
        ref_m = E.suffix_array(miss)
        okm = bool(torch.equal(slm.sa, ref_m[slm.offset:slm.offset + slm.sa.numel()]))
        out["repetitive"] = {"workload": '"mississippi$" * 10^6 (12 MB; the reference benchmark\'s text, tests/benchmark.py:110)',
                             "slices_equal_single_gpu_sa": sum_over_ranks(1.0 if okm else 0.0) == world,
                             "seconds": t_rep, "extension_rounds": slm.ext_rounds, "doubling_rounds": slm.dbl_rounds}
        assert out["repetitive"]["slices_equal_single_gpu_sa"], "distributed build of the repetitive text differs"
        del full, blk, sl, ref_sa, ref_bwt, miss, mblk, slm, ref_m
        torch.cuda.empty_cache()

        # ---- single-GPU yardstick: one rank's share (1 GB ENG96) built by the single-GPU builder on this GPU
        per_rank = min(args.dist_bytes_per_rank, int(_lib.MAX_N))
        one = torch.empty(per_rank, dtype=torch.uint8, device=dev)
        E.check(L.hkcsa_gen_text(0, 42, per_rank - 1, one.data_ptr(), torch.cuda.current_stream().cuda_stream))
        one[per_rank - 1] = 0x24
        single_ms = []
        for it in range(3):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sa1, bw1 = E.suffix_array_bwt(one)
            b.record()
            torch.cuda.synchronize()
            if it:
                single_ms.append(a.elapsed_time(b))
            del sa1, bw1
        single_ms = max_over_ranks(float(np.mean(single_ms)))
        del one
        torch.cuda.empty_cache()

        # ---- timed leg: N x 1 GB ENG96 (N = 8: the 8 GB of BASELINE configs[4])
        n_big = per_rank * world
        full, blk = make_blocks(0, 42, n_big)
        del full
        torch.cuda.empty_cache()
        sl = dist_sa.distributed_suffix_array(blk)                     # warm-up: allocates the symmetric workspace
        times = []
        for _ in range(3):
            del sl
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sl = dist_sa.distributed_suffix_array(blk)
            b.record()
            barrier()
            times.append(max_over_ranks(a.elapsed_time(b)))
        del sl
        barrier()
        sl = dist_sa.distributed_suffix_array(blk, profile=True)       # one more run, synchronised at phase boundaries
        barrier()
        ms = float(np.mean(times))
        phases = {k: max_over_ranks(v * 1e3) for k, v in sorted(sl.phases.items())}
        bytes_in = max_over_ranks(float(sl.nvlink_bytes_in))
        # ---- size-independent checks at full size
        ids = sl.sa_int64()
        m_ = ids.numel()
        g = torch.Generator(device="cpu").manual_seed(17 + rank)
        j = torch.randint(0, max(1, m_ - 1), (200_000,), generator=g).to(dev)
        bad, undecided = _suffix_order_violations(sl.text, ids[j], ids[j + 1]) if m_ > 1 else (0, 0)
        edge = torch.zeros((world, 2), dtype=torch.int64, device=dev)
        if m_:
            edge[rank, 0], edge[rank, 1] = ids[0], ids[-1]
        dist.all_reduce(edge)
        ea = edge[:-1, 1].contiguous()
        eb = edge[1:, 0].contiguous()
        bad_edge, _ = _suffix_order_violations(sl.text, ea, eb, width=4096)
        tot = torch.stack([ids.sum(), torch.tensor(m_, device=dev)])      # int64 sums wrap: compared modulo 2^64
        dist.all_reduce(tot)
        want_sum = (n_big * (n_big - 1) // 2) % (1 << 64)
        got_sum = int(tot[0].item()) % (1 << 64)
        pos = torch.where(ids[j] > 0, ids[j] - 1, torch.full_like(ids[j], n_big - 1))
        bwt_ok = bool(torch.equal(sl.bwt[j], sl.text[pos]))
        props = {"adjacent_pairs_sampled_per_rank": int(j.numel()), "order_violations": int(sum_over_ranks(float(bad))),
                 "undecided_within_96_symbols": int(sum_over_ranks(float(undecided))),
                 "slice_boundary_violations": bad_edge, "ids_sum_is_n_choose_2": got_sum == want_sum,
                 "slices_cover_n": int(tot[1].item()) == n_big,
                 "bwt_is_text_before_suffix": sum_over_ranks(1.0 if bwt_ok else 0.0) == world}
        ok_props = (props["order_violations"] == 0 and bad_edge == 0 and props["ids_sum_is_n_choose_2"]
                    and props["slices_cover_n"] and props["bwt_is_text_before_suffix"])
        out.update({
            "workload": f"{world} x {per_rank} bytes of ENG96 order-3 Markov text + '$' (BASELINE configs[4] shape"
                        + ("" if world == 8 else f", scaled to {world} GPUs") + "), SA + BWT slices",
            "text_bytes": n_big, "n_gpus": world, "suffix_id_bits": 64 if sl.sa.dtype == torch.int64 else 32,
            "ms": ms, "ms_runs": times, "MBps": n_big / 1e6 / (ms / 1e3),
            "single_gpu": {"text_bytes": per_rank, "ms": single_ms, "MBps": per_rank / 1e6 / (single_ms / 1e3),
                           "what": "hkcsa_sa_bwt_build (suffix array + BWT) of one rank's share on one GPU, same run"},
            "fraction_of_linear": (n_big / ms) / (world * per_rank / single_ms),
            "phases_ms_max_over_ranks": phases,
            "phases_note": "from one extra run that synchronises at every phase boundary (not the timed runs)",
            "rounds_rank0": sl.rounds, "extension_rounds": sl.ext_rounds, "doubling_rounds": sl.dbl_rounds,
            "nvlink": {"bytes_received_per_gpu": bytes_in, "GBps_over_whole_build": bytes_in / (ms / 1e3) / 1e9,
                       "frac_of_900GBps_over_whole_build": bytes_in / (ms / 1e3) / 1e9 / NVLINK_GBS,
                       "exchange_phase_GBps": ((bytes_in - (n_big - blk.numel())) / (phases["pack_exchange"] / 1e3) / 1e9
                                               if phases.get("pack_exchange") else None),
                       "text_allgather": "in-place all-gather left running on NCCL's stream beside the histograms, the "
                                         "exchange and the round-0 sort; phases text_allgather / text_wait = its set-up "
                                         "and what was left of it when the refinement rounds needed the text"},
            "properties_at_full_size": props, "properties_ok": ok_props,
        })
        assert ok_props, f"distributed build failed its full-size checks: {props}"
        # ---- the index the build leaves behind: per-slice wavelet trees + sampled SAs, replicated; count + locate
        barrier()
        t0 = time.perf_counter()
        ms_idx = dist_sa.replicate_sliced_index(sl, sa_sample_rate=SA_SAMPLE_RATE)
        barrier()
        t_index = max_over_ranks(time.perf_counter() - t0)
        Pq = 1_000_000
        alpha = torch.unique(sl.text[: 1 << 22])
        alpha = alpha[alpha != 0x24]
        qp, qo = E.gen_patterns(44, Pq, sl.text[: n_big - 1], alpha)
        from hkcsa import dist as hdist
        qb = hdist.shard_bounds(qo, world)[rank]
        mp, mo = hdist.local_slice(qp, qo, *qb)
        ms_idx.count_batch(mp, mo)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        qlo, qhi = ms_idx.count_batch(mp, mo)
        b.record()
        barrier()
        q_ms = max_over_ranks(a.elapsed_time(b))
        kq = min(2000, mo.numel() - 1)
        lo_off, lo_pos = ms_idx.locate_batch(mp[: int(mo[kq].item())], mo[: kq + 1])
        # every located position must hold its pattern (first 8 symbols compared on the device)
        cnt_ = (lo_off[1:] - lo_off[:-1])
        pat_of = torch.repeat_interleave(torch.arange(kq, device=dev), cnt_)
        good = True
        if lo_pos.numel():
            ar = torch.arange(8, device=dev)
            got = sl.text[(lo_pos[:, None] + ar).clamp(max=n_big - 1)]
            want = mp[(mo[:kq][pat_of][:, None] + ar)]
            good = bool(torch.equal(got, want))
        hits_match = bool(torch.equal(cnt_ > 0, qlo[:kq] >= 0))
        out["sliced_index"] = {"build_and_replicate_s": t_index, "count_patterns": Pq,
                               "count_patterns_per_s": Pq / (q_ms / 1e3), "locate_patterns_checked_per_rank": kq,
                               "located_positions_hold_the_pattern": sum_over_ranks(1.0 if good and hits_match else 0.0) == world,
                               "sa_sample_rate": SA_SAMPLE_RATE}
        assert out["sliced_index"]["located_positions_hold_the_pattern"]
    except AssertionError:
        raise
    except Exception as exc:       # e.g. symmetric memory unavailable: report instead of losing the whole line
        out["error"] = f"{type(exc).__name__}: {exc}"[:500]
    finally:
        dist_sa.release_workspaces()
    return out


# ------------------------------------------------------------------ outputs of the timed build
DUMP_ROWS = 1 << 19      # rows sampled from each length-n output: a dump stays below 40 MB at any text size
DUMP_SEED = 7


def dump_outputs(out_dir, idx):
    """Writes what one build (a DeviceIndex) hands its caller to out_dir/<name>.npy, float64 for positions and
    counts, float32 for symbols and bits, so that two builds of the project can be compared output for output.
    Outputs of length n are read at one fixed, seeded sample of DUMP_ROWS rows (every row of a smaller text):
      rows            the sampled rows, ascending
      sa, bwt         the suffix array and the BWT at those rows
      sa_via_samples  the suffix array at those rows recovered from the sampled suffix array (LF walks)
      occ             wavelet-tree rank of bwt[row] before row: the Occ value a backward-search step reads
      wt_level<l>     the bits of wavelet-tree level l at the sampled rows below that level's length
      count           C[] as (byte, number of smaller symbols), one row per symbol of the text"""
    import torch
    n = idx.n
    rows_np = (np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS
               else np.arange(n))
    rows = torch.from_numpy(rows_np.astype(np.int64)).to(idx.device)
    bwt = idx.bwt[rows]
    out = {"rows": rows_np.astype(np.float64),
           "sa": idx.sa[rows].cpu().numpy().astype(np.float64),
           "bwt": bwt.cpu().numpy().astype(np.float32),
           "sa_via_samples": idx.locate_rows(rows.to(torch.int32), use_samples=True).cpu().numpy().astype(np.float64),
           "occ": idx.wt.rank(bwt, rows).cpu().numpy().astype(np.float64)}
    for level in range(idx.wt.levels):
        m = idx.wt.level_len(level)
        out[f"wt_level{level}"] = idx.wt.bv_bits(level, 0, m)[rows[rows < m]].cpu().numpy().astype(np.float32)
    out["count"] = np.array([[ord(c), v] for c, v in idx.wt.count_table().items()], dtype=np.float64).reshape(-1, 2)
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from hkcsa import engine as E
    from hkcsa import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything libraries print meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout is redirected to stderr above, so NCCL's INFO lines (communicator ranks, NVLS, rings) land in the
        # driver's stderr log and never in the JSON line
        os.environ["NCCL_DEBUG"] = os.environ.get("HKCSA_NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        dist.init_process_group("nccl", device_id=dev)
        warm = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)               # set up the communicator
        dist.broadcast(warm, 0)
        dist.all_gather([torch.empty_like(warm) for _ in range(world)], warm)
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    kind, seed, nbytes, desc = WORKLOADS[args.workload]
    if args.size:
        nbytes = args.size
    L = _lib.load()

    # ---- synthetic text (+ '$'), resident in HBM; pinned host copy for the e2e leg
    text = torch.empty(nbytes + 1, dtype=torch.uint8, device=dev)
    E.check(L.hkcsa_gen_text(kind, seed, nbytes, text.data_ptr(), torch.cuda.current_stream().cuda_stream))
    text[nbytes] = 0x24
    n = nbytes + 1
    h_text = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_text.copy_(text)
    h_sa = torch.empty(n, dtype=torch.int32).pin_memory()
    h_bwt = torch.empty(n, dtype=torch.uint8).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    torch.cuda.synchronize()

    def build_step(src):
        return E.DeviceIndex(src, sa_sample_rate=SA_SAMPLE_RATE)

    q_idx = None
    launches0 = L.hkcsa_launch_count()
    # ---- warm-up
    idx = None
    for _ in range(args.warmup):
        idx = build_step(text)
    torch.cuda.synchronize()
    launches_per_step = (L.hkcsa_launch_count() - launches0) // max(1, args.warmup)

    # ---- timed: K device-resident builds, CUDA events per step, L2 flushed between steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    E.prof_enable(True, classes=[TOP_KERNEL_CLASS])    # live durations of the dominant kernel only (roofline)
    clk = ClockSampler(local)          # samples through both timed regions (device-resident and e2e)
    clk.__enter__()
    barrier()
    wall0 = time.perf_counter()
    for a, b in ev:
        flush.zero_()
        a.record()
        idx = build_step(text)
        b.record()
    barrier()
    wall = time.perf_counter() - wall0
    prof_top = E.prof_read()
    E.prof_enable(False)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    ms = max_over_ranks(float(np.mean(step_ms)))
    value = world * nbytes / 1e6 / (ms / 1e3)
    stats = idx.stats.sa
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, idx)

    # ---- e2e: host text -> H2D -> build -> D2H of the INDEX (wavelet-tree blob + sampled-SA blob: what a build
    #      produces and what save() / a serving process needs), every step.  The full suffix array (4n bytes) is an
    #      on-demand product: e2e_full_sa below ships it and the BWT as well.
    h_wt = torch.empty(int(idx.wt.blob.numel()), dtype=torch.uint8).pin_memory()
    h_ssa = torch.empty(int(idx.ssa.blob.numel()), dtype=torch.uint8).pin_memory()
    try:        # pinned buffers are first touched by this thread: keep it on the CPUs next to this GPU
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass

    def e2e_step(full_sa: bool):
        d = torch.empty(n, dtype=torch.uint8, device=dev)
        d.copy_(h_text, non_blocking=True)
        if full_sa:
            ix = E.DeviceIndex(d, sa_sample_rate=SA_SAMPLE_RATE, host_sa=h_sa, host_bwt=h_bwt)
        else:
            ix = E.DeviceIndex(d, sa_sample_rate=SA_SAMPLE_RATE, keep_sa=False)
            h_wt.copy_(ix.wt.blob, non_blocking=True)
            h_ssa.copy_(ix.ssa.blob, non_blocking=True)
        torch.cuda.synchronize()      # build + device->host copies done
        return ix

    def time_e2e(full_sa: bool):
        e2e_step(full_sa)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()
            e2e_step(full_sa)
        barrier()
        return max_over_ranks((time.perf_counter() - t0) / args.steps * 1e3)

    e2e_ms = time_e2e(False)
    e2e_value = world * nbytes / 1e6 / (e2e_ms / 1e3)
    e2e_full_ms = time_e2e(True)
    clk.__exit__(None, None, None)
    e2e_d2h = int(h_wt.numel() + h_ssa.numel())

    # ---- e2e through the drop-in API: a Python str in, numpy answers out (rank 0, N = 1 only)
    e2e_api = None
    if world == 1 and not args.no_queries:
        from csa.enhanced_fm_index import EnhancedFMIndex
        s_text = h_text.numpy()[:nbytes].tobytes().decode("latin-1")
        EnhancedFMIndex(s_text[: 1 << 20])                   # first call: staging buffer, module imports
        t_api = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fm = EnhancedFMIndex(s_text)
            torch.cuda.synchronize()
            t_api.append(time.perf_counter() - t0)
        rng = np.random.RandomState(5)
        starts_ = rng.randint(0, nbytes - 64, size=100_000)
        lens_ = rng.randint(8, 65, size=100_000)
        qs = [s_text[a:a + b] for a, b in zip(starts_.tolist(), lens_.tolist())]
        fm.find_range_batch(qs[:1000])
        t0 = time.perf_counter()
        lo_a, hi_a = fm.find_range_batch(qs)
        t_q = time.perf_counter() - t0
        assert isinstance(lo_a, np.ndarray) and bool((lo_a >= 0).all())
        e2e_api = {"what": "EnhancedFMIndex(str) -> find_range_batch(list[str]) -> numpy, wall clock: the str's bytes staged "
                           "through the library's pinned ring (hkcsa_h2d_staged), build, pattern packing, D2H",
                   "build_ms": 1e3 * float(np.min(t_api)), "build_MBps": nbytes / 1e6 / float(np.min(t_api)),
                   "queries": len(qs), "find_range_batch_ms": 1e3 * t_q, "patterns_per_s": len(qs) / t_q}
        del fm, s_text, qs

    # ---- per-kernel breakdown: two more builds with every kernel class timed (outside the timed region: the
    #      event pairs around ~130 launches per build are not free)
    E.prof_enable(True)
    for _ in range(2):
        flush.zero_()
        build_step(text)
    prof = E.prof_read()
    E.prof_enable(False)
    for v in prof.values():
        v["steps"] = 2
    prof[TOP_KERNEL_CLASS] = prof_top[TOP_KERNEL_CLASS]     # the roofline kernel: from the timed region itself
    prof[TOP_KERNEL_CLASS]["steps"] = args.steps

    # ---- dominant kernel roofline: onesweep radix pass, 24 B per (key, value) pair per launch
    peak, peak_src = measured_peak_gbs()
    top = max(prof.items(), key=lambda kv: kv[1]["ms"] / kv[1]["steps"]) if prof else (None, None)
    one = prof.get("onesweep_u64")
    roofline = None
    traffic = None
    try:   # DRAM bytes per pair from the committed ncu --set full capture, scaled to this run's average launch
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)["onesweep64_kernel"]
        per_pair = (tr["dram_bytes_read"] + tr["dram_bytes_write"]) / tr["pairs_in_profiled_launch"]
        if one and one["launches"]:
            traffic = per_pair * (one["alg_bytes"] / 24.0) / one["launches"]
    except Exception:
        traffic = None
    if one and one["ms"] > 0:
        achieved = one["alg_bytes"] / (one["ms"] / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": "onesweep64_kernel (one 8-bit LSD radix pass, 24 B per (u64,u32) pair)",
                    "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "traffic_source": "profiles/r02_traffic.json: dram bytes per pair of one ncu --set full capture of this "
                                      "kernel, scaled to this run's average launch (not measured in this run)",
                    "alg_bytes_per_launch": one["alg_bytes"] / one["launches"],
                    "launches": one["launches"], "avg_launch_ms": one["ms"] / one["launches"],
                    "share_of_step": one["ms"] / max(1e-9, sum(step_ms))}

    # ---- batched count / locate (BASELINE config 4 shape).  N > 1: rank 0's index is broadcast over
    #      NCCL, the SAME global batch is cut into contiguous slices balanced by total symbols
    #      (hkcsa.dist.shard_bounds), every rank searches its slice, (lo, hi) are all-gathered.
    queries = None
    if not args.no_queries and args.patterns > 0:
        from hkcsa import dist as hdist
        P_total = args.patterns
        alpha = torch.from_numpy(np.frombuffer(idx.wt.alphabet, dtype=np.uint8).copy()).to(dev)
        alpha = alpha[alpha != 0x24]
        pats, off = E.gen_patterns(44, P_total, text[:nbytes], alpha)       # identical on every rank
        bcast_ms = None
        q_idx = idx
        if world > 1:
            barrier()
            t0 = time.perf_counter()
            q_idx = hdist.broadcast_index(idx if rank == 0 else None, src=0, device=dev, with_bwt=True)
            barrier()
            bcast_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
            bounds = hdist.shard_bounds(off, world)
            pb, pe = bounds[rank]
            my_pats, my_off = hdist.local_slice(pats, off, pb, pe)
        else:
            my_pats, my_off = pats, off
        P = my_off.numel() - 1
        torch.cuda.synchronize()
        reps = 3

        def time_count(use_table, use_occ=False):
            for _ in range(2):
                q_idx.count_batch(my_pats, my_off, use_kmer_table=use_table, use_occ_table=use_occ)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                r_ = q_idx.count_batch(my_pats, my_off, use_kmer_table=use_table, use_occ_table=use_occ)
            b.record()
            barrier()
            return max_over_ranks(a.elapsed_time(b) / reps), r_

        c_ms_plain, (lo0, hi0) = time_count(False)          # every symbol walks the wavelet tree
        t0 = time.perf_counter()
        q_idx.build_kmer_table()
        torch.cuda.synchronize()
        kmer_ms = (time.perf_counter() - t0) * 1e3
        c_ms, (lo, hi) = time_count(True)                   # last k symbols from the k-mer jump table
        assert torch.equal(lo, lo0) and torch.equal(hi, hi0)
        occ_info = None
        if q_idx.bwt is not None:          # same queries ranked on the sampled Occ table (identical ranges)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            plan_o, _ = q_idx.build_occ_table(5, layout=1)
            torch.cuda.synchronize()
            occ_build_ms = (time.perf_counter() - t0) * 1e3
            o_ms, (lo_o, hi_o) = time_count(True, True)
            assert torch.equal(lo, lo_o) and torch.equal(hi, hi_o)
            occ_info = {"count_patterns_per_s": P_total / (o_ms / 1e3), "count_ms": o_ms, "build_ms": occ_build_ms,
                        "bytes": int(plan_o.blob_bytes), "layout": "per-symbol bitmaps, one 8-byte entry per 32 rows"}
            q_idx._occ = None
        gather_ms = None
        if world > 1:                      # results to every rank, timed apart from the search
            hdist.gather_ranges(lo, hi, bounds)                      # first call: NCCL channel set-up
            barrier()
            t0 = time.perf_counter()
            glo, ghi = hdist.gather_ranges(lo, hi, bounds)
            barrier()
            gather_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
            hits = float((glo >= 0).sum().item())
        else:
            hits = float((lo >= 0).sum().item())
        # locate a slice of this rank's patterns through the sampled SA (LF walks)
        PL = min(P, 1_000_000 // world)
        offL = my_off[: PL + 1]
        a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o_off, o_pos = q_idx.locate_batch(my_pats, offL, use_samples=True)
        torch.cuda.synchronize()
        a2.record()
        o_off, o_pos = q_idx.locate_batch(my_pats, offL, use_samples=True)
        b2.record()
        barrier()
        l_ms = max_over_ranks(a2.elapsed_time(b2))
        occ_total = sum_over_ranks(float(o_pos.numel()))
        best_ms = min(c_ms, occ_info["count_ms"]) if occ_info else c_ms
        queries = {"count_patterns_per_s": P_total / (best_ms / 1e3), "count_patterns": P_total,
                   "count_ms": best_ms,
                   "rank_structure": ("sampled Occ table (per-symbol bitmaps)" if occ_info and occ_info["count_ms"] < c_ms
                                      else "wavelet tree") + " + k-mer jump table",
                   "count_patterns_per_s_wavelet_tree": P_total / (c_ms / 1e3),
                   "hit_fraction": hits / P_total, "pattern_len": "uniform 8-64",
                   "count_patterns_per_s_no_jump_table": P_total / (c_ms_plain / 1e3),
                   "occ_table": occ_info,
                   "kmer_jump_table": {"k": int(q_idx._kmer[1]), "build_ms": kmer_ms,
                                       "bytes": int(q_idx._kmer[0].numel() * 4) if q_idx._kmer[0] is not None else 0},
                   "index_broadcast_ms": bcast_ms, "result_allgather_ms": gather_ms,
                   "locate_occurrences_per_s": occ_total / (l_ms / 1e3), "locate_patterns": PL * world,
                   "locate_occurrences": occ_total, "locate_ms": l_ms, "sa_sample_rate": SA_SAMPLE_RATE,
                   "scaling": "strong (fixed global batch)",
                   "sharding": "index broadcast from rank 0, patterns split into contiguous slices balanced by symbols"}

    # ---- BASELINE configs[2] and [3]: the 200 MB English-like text.  Every rank builds the index (replicas: C3 is a
    #      single-GPU build), timed like the headline; then 10 M count queries, patterns sharded over the ranks.
    c3 = None
    c4 = None
    if not args.no_c3 and args.workload == "c2" and not args.size:
        from hkcsa import dist as hdist
        k3, s3, n3, d3 = WORKLOADS["c3"]
        idx = q_idx = None
        torch.cuda.empty_cache()
        t3 = torch.empty(n3 + 1, dtype=torch.uint8, device=dev)
        E.check(L.hkcsa_gen_text(k3, s3, n3, t3.data_ptr(), torch.cuda.current_stream().cuda_stream))
        t3[n3] = 0x24
        idx3 = None
        for _ in range(3):                       # warm-up: the caching allocator settles on this size class
            idx3 = E.DeviceIndex(t3, sa_sample_rate=SA_SAMPLE_RATE)
        torch.cuda.synchronize()
        ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(8)]
        E.prof_enable(True, classes=[TOP_KERNEL_CLASS])
        barrier()
        for a, b in ev3:
            flush.zero_()
            a.record()
            idx3 = E.DeviceIndex(t3, sa_sample_rate=SA_SAMPLE_RATE)
            b.record()
        barrier()
        p3 = E.prof_read().get(TOP_KERNEL_CLASS)
        E.prof_enable(False)
        # median: this record runs late in the process, with the caching allocator full of the earlier legs' blocks,
        # and an occasional step pays a cudaMalloc / cudaFree round trip (the per-step list is in the record)
        c3_mine = float(np.median([a.elapsed_time(b) for a, b in ev3]))
        c3_ms = max_over_ranks(c3_mine)
        c3_all = [c3_mine]
        if world > 1:
            t_all = torch.zeros(world, dtype=torch.float64, device=dev)
            t_all[rank] = c3_mine
            dist.all_reduce(t_all)
            c3_all = [round(v, 3) for v in t_all.cpu().tolist()]
        st3 = idx3.stats.sa
        c3 = {"workload": d3, "text_bytes": n3, "steps": len(ev3), "warmup": 3, "ms_per_step": c3_ms,
              "ms_per_step_is": "median over the steps, max over ranks",
              "ms_steps_this_rank": [round(a.elapsed_time(b), 3) for a, b in ev3], "ms_per_rank": c3_all,
              "value_MBps": world * n3 / 1e6 / (c3_ms / 1e3),
              "roofline_onesweep": ({"achieved": p3["alg_bytes"] / (p3["ms"] / 1e3) / 1e9, "peak": peak,
                                     "frac": p3["alg_bytes"] / (p3["ms"] / 1e3) / 1e9 / peak, "launches": p3["launches"],
                                     "share_of_step": p3["ms"] / (len(ev3) * c3_mine)} if p3 and p3["ms"] > 0 else None),
              "sa": {"rounds": int(st3.rounds), "k0": int(st3.k0),
                     "round_elems": [int(st3.round_elems[i]) for i in range(int(st3.rounds))],
                     "round_passes": [int(st3.round_passes[i]) for i in range(int(st3.rounds))]},
              "wavelet_levels": idx3.wt.levels, "index_bytes": int(idx3.wt.blob.numel() + idx3.ssa.blob.numel())}
    if c3 is not None and not args.no_queries and args.patterns > 0:
        alpha3 = torch.from_numpy(np.frombuffer(idx3.wt.alphabet, dtype=np.uint8).copy()).to(dev)
        alpha3 = alpha3[alpha3 != 0x24]
        pats3, off3 = E.gen_patterns(44, args.patterns, t3[:n3], alpha3)
        pats3_full, off3_full = pats3, off3
        total_syms3 = int(pats3_full.numel())
        bounds3 = hdist.shard_bounds(off3_full, world)
        if world > 1:
            pb, pe = bounds3[rank]
            pats3, off3 = hdist.local_slice(pats3, off3, pb, pe)
        idx3.build_kmer_table()

        def time_count3(use_occ):
            for _ in range(2):
                idx3.count_batch(pats3, off3, use_kmer_table=True, use_occ_table=use_occ)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                r_ = idx3.count_batch(pats3, off3, use_kmer_table=True, use_occ_table=use_occ)
            b.record()
            barrier()
            return max_over_ranks(a.elapsed_time(b) / 3), r_

        c4_ms, (lo3, hi3) = time_count3(False)
        kk3 = int(idx3._kmer[1])
        steps3 = total_syms3 - kk3 * args.patterns          # rank steps if every pattern walked all its symbols
        c4 = {"workload": "10 M count queries (len 8-64) on the 200 MB ENG96 index (BASELINE configs[3])",
              "count_patterns_per_s": args.patterns / (c4_ms / 1e3), "count_ms": c4_ms,
              "hit_fraction": sum_over_ranks(float((lo3 >= 0).sum().item())) / args.patterns,
              "rank_structure": "wavelet tree + k-mer jump table",
              "wavelet_levels": idx3.wt.levels, "kmer_k": kk3}

        def roofline_q(ms_, requests_per_step, what):
            req = float(steps3) * requests_per_step
            return {"structure": what, "bound": "hbm random 32-byte sectors",
                    "alg_requests": req, "alg_bytes": req * 32.0, "alg_bytes_per_pattern": req * 32.0 / args.patterns,
                    "requests_per_s": req / (ms_ / 1e3), "achieved": req * 32.0 / (ms_ / 1e3) / 1e9, "peak": peak,
                    "unit": "GB/s", "frac": req * 32.0 / (ms_ / 1e3) / 1e9 / peak,
                    "note": "upper bound on the work: 2 boundaries x (pattern symbols - k) x requests per rank x 32 B; "
                            "misses stop early and narrow ranges share a sector, so the true request count is lower"}

        c4["roofline_queries"] = [roofline_q(c4_ms, 2.0 * idx3.wt.levels, "wavelet tree: one sector per level per boundary")]
        # locate of the first 1 M patterns of this rank through the sampled SA (LF walks)
        PL3 = min(off3.numel() - 1, 1_000_000 // world)

        def time_locate3():
            idx3.locate_batch(pats3, off3[: PL3 + 1], use_samples=True)
            torch.cuda.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            _, pos_ = idx3.locate_batch(pats3, off3[: PL3 + 1], use_samples=True)
            b_.record()
            barrier()
            return max_over_ranks(a_.elapsed_time(b_)), sum_over_ranks(float(pos_.numel()))

        l3_ms, l3_occ = time_locate3()
        c4["locate_occurrences_per_s"] = l3_occ / (l3_ms / 1e3)
        c4["locate_ms"] = l3_ms
        c4["locate_occurrences"] = l3_occ
        c4["roofline_locate"] = {"bound": "hbm random 32-byte sectors", "sa_sample_rate": SA_SAMPLE_RATE,
                                 "alg_requests": l3_occ * (SA_SAMPLE_RATE - 1) / 2.0 * (idx3.wt.levels + 1),
                                 "note": "expected (rate-1)/2 LF steps per occurrence x (levels + 1 mark block) sectors"}
        c4["roofline_locate"]["achieved"] = c4["roofline_locate"]["alg_requests"] * 32.0 / (l3_ms / 1e3) / 1e9
        c4["roofline_locate"]["frac"] = c4["roofline_locate"]["achieved"] / peak
        # the same queries ranked on the sampled Occ table (second rank structure, identical ranges)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plan_o, blob_o = idx3.build_occ_table(5, layout=1)
        torch.cuda.synchronize()
        occ_ms = (time.perf_counter() - t0) * 1e3
        o_ms, (lo4, hi4) = time_count3(True)
        assert torch.equal(lo4, lo3) and torch.equal(hi4, hi3)
        lo_ms, lo_occ = time_locate3()
        c4["occ_table_bitmaps"] = {"count_patterns_per_s": args.patterns / (o_ms / 1e3), "count_ms": o_ms,
                                   "build_ms": occ_ms, "bytes": int(plan_o.blob_bytes),
                                   "locate_occurrences_per_s": lo_occ / (lo_ms / 1e3), "locate_ms": lo_ms}
        c4["roofline_queries"].append(roofline_q(o_ms, 2.0, "sampled Occ table (bitmaps): one 8-byte entry = one request per rank"))
        c4["count_patterns_per_s_wavelet_tree"] = c4["count_patterns_per_s"]
        if o_ms < c4_ms:
            c4["count_patterns_per_s"] = args.patterns / (o_ms / 1e3)
            c4["count_ms"] = o_ms
            c4["rank_structure"] = "sampled Occ table (per-symbol bitmaps) + k-mer jump table"
        if world > 1:
            # every rank needs every answer.  (a) search + NCCL all-gather of int64 (lo, hi); (b) the search in chunks
            # with a store kernel pushing packed 8-byte answers into the symmetric result array of every rank
            # (unicast peer stores, and multimem.st through the NVSwitch multicast mapping when there is one)
            def timed3(fn):
                fn()
                torch.cuda.synchronize()
                barrier()
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                for _ in range(5):
                    r_ = fn()
                b_.record()
                torch.cuda.synchronize()
                barrier()
                return max_over_ranks(a_.elapsed_time(b_) / 5), r_

            def nccl3():
                l_, h_ = idx3.count_batch(pats3, off3, use_kmer_table=True, use_occ_table=True)
                return hdist.gather_ranges(l_, h_, bounds3)

            g_ms, (glo3, ghi3) = timed3(nccl3)
            allr = {"search_plus_nccl_allgather": {"ms": g_ms, "patterns_per_s": args.patterns / (g_ms / 1e3),
                                                  "bytes_per_pattern": 16}}
            try:
                for label, mc in (("search_plus_peer_store_gather", False), ("search_plus_multimem_store_gather", True)):
                    try:
                        pg = hdist.PeerGather(args.patterns, dev, use_multicast=mc)
                    except RuntimeError as exc:
                        allr[label] = {"unavailable": str(exc)[:200]}
                        continue
                    best = None
                    for chunks in (1, 4, 8):
                        sl3 = hdist.chunked_slices(pats3_full, off3_full, bounds3[rank][0], bounds3[rank][1], chunks)
                        f_ms, packed = timed3(lambda: hdist.sharded_count_packed(idx3, sl3, pg, use_kmer_table=True,
                                                                                 use_occ_table=True))
                        plo, phi = pg.unpack()
                        assert torch.equal(plo, glo3) and torch.equal(phi, ghi3), "packed gather differs from NCCL gather"
                        if best is None or f_ms < best["ms"]:
                            best = {"ms": f_ms, "patterns_per_s": args.patterns / (f_ms / 1e3), "chunks": chunks,
                                    "bytes_per_pattern": 8, "identical_to_nccl_gather": True}
                    allr[label] = best
                    del pg
            except Exception as exc:       # symmetric memory unavailable on this box: report, do not fail
                allr["peer_store_gather_error"] = f"{type(exc).__name__}: {exc}"[:300]
            allr["note"] = ("device time (CUDA events, max over ranks) of search + delivery of all 10 M answers to every "
                            "rank, incl. the cross-rank barriers of the store path")
            c4["all_answers_on_all_ranks"] = allr
        del blob_o
        idx3._occ = None

    # ---- BASELINE configs[4]: distributed suffix-array + BWT build (N > 1), N x 1 GB of ENG96 text
    dist_build = None
    if world > 1 and not args.no_dist_build:
        # free the replicas' indexes, texts and pattern batches: the distributed legs need the memory
        idx = q_idx = idx3 = t3 = pats3 = off3 = pats3_full = off3_full = pats = off = my_pats = my_off = None
        lo = hi = lo0 = hi0 = lo3 = hi3 = lo4 = hi4 = glo3 = ghi3 = o_off = o_pos = text = flush = None
        torch.cuda.empty_cache()
        dist_build = run_dist_build(args, world, rank, dev, barrier, max_over_ranks, sum_over_ranks, peak)

    # ---- CPU baseline (rank 0, N = 1 only): oracle port on a bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = min(nbytes, args.cpu_sample)
        dt, threads, _ = cpu_build_sample(kind, seed, sample)
        cpu = {"value": sample / 1e6 / dt, "unit": "MB/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} bytes of the workload text (+'$'): oracle port of SA+BWT+WT spine, "
                         f"{dt:.2f} s on {threads} threads"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 symbols / u32 ranks / u64 keys (integer)", "data": "synthetic",
            "config": {"workload": desc, "text_bytes": nbytes, "index_symbols": n, "sa_sample_rate": SA_SAMPLE_RATE,
                       "parallelism": f"replicas x{world}" if world > 1 else "single GPU",
                       "l2": "256 MiB flush buffer written between timed steps; working set >> L2"},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": "MB/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": n,
                    "d2h_bytes_per_step": e2e_d2h,
                    "what": "pinned host text -> H2D -> build -> D2H of the index (wavelet-tree blob + sampled-SA "
                            "blob), wall clock incl. final sync; the full suffix array is shipped by e2e_full_sa"},
            "e2e_full_sa": {"value": world * nbytes / 1e6 / (e2e_full_ms / 1e3), "unit": "MB/s", "ms_per_step": e2e_full_ms,
                            "h2d_bytes_per_step": n, "d2h_bytes_per_step": 5 * n,
                            "what": "the same with D2H of SA (4n) + BWT (n) as well (what round 1 shipped)"},
            "e2e_api": e2e_api,
            "gpu_launches": int(launches_per_step) * args.steps,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "kernels": {k: {"ms_per_step": v["ms"] / v["steps"], "launches_per_step": v["launches"] / v["steps"],
                            "alg_GBps": (v["alg_bytes"] / (v["ms"] / 1e3) / 1e9) if v["ms"] > 0 and v["alg_bytes"] else None}
                        for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"] / kv[1]["steps"])},
            "kernels_note": TOP_KERNEL_CLASS + ": CUDA events inside the timed region; the other classes: two extra "
                            "builds after it with every launch bracketed",
            "top_kernel": top[0],
            "sa": {"rounds": int(stats.rounds), "k0": int(stats.k0), "bits_per_symbol": int(stats.bits_per_symbol),
                   "round_elems": [int(stats.round_elems[i]) for i in range(int(stats.rounds))],
                   "round_passes": [int(stats.round_passes[i]) for i in range(int(stats.rounds))],
                   "alg_bytes": int(stats.alg_bytes)},
            "queries": queries,
            "c3": c3,
            "queries_c4": c4,
            "dist_build": dist_build,
            "wall_s_timed_region": wall,
        }
        sys.stdout.flush()
        # the one JSON line goes to the REAL stdout; fd 1 stays pointed at stderr so that whatever NCCL logs while the
        # process group is torn down cannot follow the line
        os.write(saved_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
