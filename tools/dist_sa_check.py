"""torchrun check of the distributed suffix-array build (hkcsa.dist_sa) on real GPUs:
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/dist_sa_check.py [--size BYTES] [--kind 0|1] [--verify]
Every rank contributes a contiguous block of the synthetic text; the slices are gathered on rank 0 and, with
--verify, compared with the single-GPU builder.  Prints one JSON line with the timing (max over ranks)."""
import argparse, json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "high-order-entropy-compressed-suffix-array_b200"))
import numpy as np, torch, torch.distributed as dist
from hkcsa import engine as E, dist_sa

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=50_000_000)
ap.add_argument("--kind", type=int, default=0)
ap.add_argument("--verify", action="store_true")
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--patterns", type=int, default=1_000_000)
ap.add_argument("--wide", action="store_true", help="force 64-bit suffix ids (automatic beyond 2^32-2 symbols)")
ap.add_argument("--sa-only", action="store_true", help="stop after the suffix array / BWT check")
ap.add_argument("--profile", action="store_true", help="synchronise at phase boundaries and report seconds per phase")
ap.add_argument("--props", action="store_true", help="size-independent checks (no single-GPU reference: n may exceed 2^30)")
args = ap.parse_args()
world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
os.environ.setdefault("NCCL_DEBUG", "WARN")
dist.init_process_group("nccl", device_id=dev)
n = args.size
if args.kind == 2:                                              # the reference benchmark's workload (tests/benchmark.py:110), scaled
    reps_ = n // 12
    n = reps_ * 12
    full = torch.from_numpy(np.frombuffer(b"mississippi$" * reps_, dtype=np.uint8).copy()).to(dev)
elif args.kind == 3:                                            # a 1 MB English-like block repeated: LCPs of megabytes
    unit = E.gen_text(0, 7, 1 << 20)
    full = unit.repeat(-(-n // (1 << 20)))[:n].contiguous()
    full[n - 1] = 0x24
else:
    full = E.gen_text(args.kind, 42 + args.kind, n)             # same bytes on every rank; keep only my block
    full[n - 1] = 0x24                                          # unique sentinel (the generators never emit '$'): LF walks need it
lo, hi = n * rank // world, n * (rank + 1) // world
block = full[lo:hi].clone()
del full
torch.cuda.synchronize(); dist.barrier()
best = None
for _ in range(args.reps):
    torch.cuda.synchronize(); dist.barrier(); t0 = time.perf_counter()
    sl = dist_sa.distributed_suffix_array(block, wide=True if args.wide else None, profile=args.profile)
    torch.cuda.synchronize(); dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    best = float(dt.item()) if best is None else min(best, float(dt.item()))
counts = torch.zeros(world, dtype=torch.int64, device=dev); counts[rank] = sl.sa.numel()
dist.all_reduce(counts)
ok = None
if args.verify:
    cmax = int(counts.max().item())
    pad = torch.zeros(cmax, dtype=torch.int32, device=dev); pad[: sl.sa.numel()] = sl.sa.to(torch.int32)
    bpad = torch.zeros(cmax, dtype=torch.uint8, device=dev); bpad[: sl.bwt.numel()] = sl.bwt
    gs = [torch.empty_like(pad) for _ in range(world)]; gb = [torch.empty_like(bpad) for _ in range(world)]
    dist.all_gather(gs, pad); dist.all_gather(gb, bpad)
    if rank == 0:
        sa = torch.cat([gs[r][: int(counts[r])] for r in range(world)])
        bw = torch.cat([gb[r][: int(counts[r])] for r in range(world)])
        ref = E.suffix_array(sl.text)
        ok = bool(torch.equal(sa, ref)) and bool(torch.equal(bw, E.bwt(sl.text, ref)))
if args.sa_only:
    if rank == 0:
        print(json.dumps({"check": "distributed_suffix_array", "world": world, "text_bytes": n, "kind": args.kind,
                          "seconds": best, "MB_per_s": n / 1e6 / best, "slice_sizes": counts.cpu().tolist(),
                          "rounds": sl.rounds, "ext_rounds": sl.ext_rounds, "dbl_rounds": sl.dbl_rounds,
                          "phases_s_rank0": sl.phases, "nvlink_bytes_in_rank0": sl.nvlink_bytes_in,
                          "verified_against_single_gpu": ok}), flush=True)
    dist.destroy_process_group()
    sys.exit(0)
# ---- the index the distributed build leaves behind: per-slice wavelet trees + sampled SAs, replicated on every
#      rank, then the pattern batch is sharded (config 4 style) over the ranks
from hkcsa import dist as hdist
torch.cuda.synchronize(); dist.barrier(); t0 = time.perf_counter()
ms = dist_sa.replicate_sliced_index(sl, sa_sample_rate=32)
torch.cuda.synchronize(); dist.barrier()
t_index = time.perf_counter() - t0
P = args.patterns
alpha = torch.unique(sl.text[: min(n, 1 << 22)])
pats, off = E.gen_patterns(44, P, sl.text, alpha)
bounds = hdist.shard_bounds(off.cpu().numpy(), world)
my_p, my_o = hdist.local_slice(pats, off, *bounds[rank])
lo, hi = ms.count_batch(my_p, my_o)
torch.cuda.synchronize(); dist.barrier()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); lo, hi = ms.count_batch(my_p, my_o); b.record(); torch.cuda.synchronize()
cms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev); dist.all_reduce(cms, op=dist.ReduceOp.MAX)
q_ok = None
if args.verify:
    glo, ghi = hdist.sharded_count(lambda p_, o_: (lo, hi), pats, off)
    o2, p2 = ms.locate_batch(my_p[: int(my_o[min(2000, my_o.numel() - 1)])], my_o[: min(2000, my_o.numel() - 1) + 1])
    if rank == 0:
        txt = torch.cat([sl.text, torch.tensor([], dtype=torch.uint8, device=dev)])
        one = E.DeviceIndex(txt, sa_sample_rate=0)
        wlo, whi = one.count_batch(pats, off)
        q_ok = bool(torch.equal(glo, wlo)) and bool(torch.equal(ghi, whi))
        o1, p1 = one.locate_batch(my_p[: int(my_o[min(2000, my_o.numel() - 1)])], my_o[: min(2000, my_o.numel() - 1) + 1],
                                  use_samples=False)
        q_ok = q_ok and bool(torch.equal(o1, o2)) and bool(torch.equal(p1.to(torch.int64) & 0xFFFFFFFF, p2))
props_ok = None
if args.props:
    # ranks 0 and world/2 (host RAM: the text is copied back): the slice is sorted (adjacent suffixes compared on
    # a sample) and located positions hold the pattern
    import random
    checker = rank in (0, world // 2)
    h_text = sl.text.cpu().numpy() if checker else None
    ids = sl.sa_int64().cpu().numpy() if checker else []
    rnd = random.Random(rank)
    good = True
    for _ in range(20000 if checker else 0):
        j = rnd.randrange(max(1, len(ids) - 1))
        if j + 1 < len(ids):
            a_, b_ = int(ids[j]), int(ids[j + 1])
            good &= h_text[a_:a_ + 256].tobytes() <= h_text[b_:b_ + 256].tobytes()   # 256-byte prefixes, in order
    k = min(2000, my_o.numel() - 1) if checker else 0
    oo, pp = ms.locate_batch(my_p[: int(my_o[k])], my_o[: k + 1])
    oo, pp = oo.cpu().numpy(), pp.cpu().numpy()
    hp, ho = my_p.cpu().numpy(), my_o.cpu().numpy()
    clo = lo.cpu().numpy()
    for q in range(k):
        m_ = int(ho[q + 1] - ho[q])
        if 0x24 in hp[ho[q]:ho[q + 1] - 1]:                     # backward search counts a '$' step inside a pattern
            continue                                            # across the text's end too (kind 2: '$' recurs)
        occ = pp[oo[q]:oo[q + 1]]
        good &= (len(occ) > 0) == (clo[q] >= 0)
        for x in occ[:4]:
            good &= h_text[int(x):int(x) + m_].tobytes() == hp[ho[q]:ho[q + 1]].tobytes()
    flag = torch.tensor([1 if good else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    props_ok = bool(flag.item())
if rank == 0:
    print(json.dumps({"check": "distributed_suffix_array", "world": world, "text_bytes": n, "kind": args.kind,
                      "seconds": best, "MB_per_s": n / 1e6 / best, "slice_sizes": counts.cpu().tolist(),
                      "rounds": sl.rounds, "ext_rounds": sl.ext_rounds, "dbl_rounds": sl.dbl_rounds,
                      "phases_s_rank0": sl.phases, "nvlink_bytes_in_rank0": sl.nvlink_bytes_in,
                      "verified_against_single_gpu": ok,
                      "sliced_index_build_and_replicate_s": t_index, "count_patterns": P,
                      "count_patterns_per_s": P / (float(cms.item()) / 1e3),
                      "queries_verified_against_single_gpu": q_ok, "property_checks": props_ok}), flush=True)
dist.destroy_process_group()
