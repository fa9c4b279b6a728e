"""Distributed suffix-array build for texts beyond one GPU's working set (SURVEY.md section 8e,
BASELINE config 5).  One process per GPU; csrc/dist_sa.cu holds the kernels.

    1. every rank holds a contiguous block of the text; the blocks are all-gathered over NCCL (one collective on
       equal blocks) so that every GPU has the whole text -- the BWT gather needs it anyway;
    2. byte histogram -> the same round-0 prefix code on every rank; every rank histograms the top 16 key bits of
       the suffixes of ITS block; the histograms are all-gathered and every rank derives the same balanced cut
       points and the (source, destination) count matrix;
    3. the all-to-all bucket exchange: the pack kernel stores each (key, suffix id) straight into the receive
       arrays of the rank owning its bucket -- symmetric memory, peer-mapped over NVLink, no collective;
    4. every rank radix-sorts what it received and refines: extension rounds on the replicated text, then -- for
       repetitive texts -- rank doubling through the ranks' peer-mapped ISA blocks (any text is sorted);
    5. the slices, concatenated in rank order, are the suffix array; the BWT slice is a local gather.

The per-rank program is a generator that yields its collective steps, so the same code runs under
torch.distributed (`distributed_suffix_array`) and with the ranks emulated in one process on one GPU
(`emulate_distributed_suffix_array`: what the single-GPU tests run).
"""
from __future__ import annotations

import ctypes as C
import os
import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from ._lib import DsaPlan, check
from .engine import _empty, _expand_ranges, _extract_requests, _ptr, _scratch, _stream, byte_hist

EXT_ROUNDS_MAX = 6          # extension rounds before rank doubling takes over


def balanced_bucket_ranges(bucket_hist: np.ndarray, parts: int) -> list[tuple[int, int]]:
    """Cut the bucket axis into `parts` contiguous ranges with near-equal suffix counts (host logic)."""
    h = np.asarray(bucket_hist, dtype=np.int64)
    nb = len(h)
    cum = np.concatenate([[0], np.cumsum(h)])
    total = int(cum[-1])
    cuts = [0]
    for r in range(1, parts):
        target = (total * r) // parts
        c = int(np.searchsorted(cum, target, side="left"))
        cuts.append(min(nb, max(c, cuts[-1])))
    cuts.append(nb)
    return [(cuts[r], cuts[r + 1]) for r in range(parts)]


def exchange_layout(hist_all: np.ndarray, parts: int):
    """hist_all[src][bucket] -> (cuts[parts+1], cnt[src][dst], counts[dst], slice_off[parts+1]): the same on every
    rank.  Source `s` writes its pairs for destination `d` from slot cnt[:s, d].sum() on."""
    hist_all = np.asarray(hist_all, dtype=np.int64)
    ranges = balanced_bucket_ranges(hist_all.sum(0), parts)
    cuts = np.array([r[0] for r in ranges] + [hist_all.shape[1]], dtype=np.int64)
    cnt = np.stack([hist_all[:, a:b].sum(1) for a, b in ranges], axis=1)        # [src][dst]
    counts = cnt.sum(0)
    slice_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return cuts, cnt, counts, slice_off


def exchange_layout_from_counts(cuts, cnt: np.ndarray):
    """The same from cut points chosen on a sampled histogram and the exact cnt[src][dst] counted under them."""
    cnt = np.asarray(cnt, dtype=np.int64)
    counts = cnt.sum(0)
    slice_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return np.asarray(cuts, dtype=np.int64), cnt, counts, slice_off


EDGE_HEAD, EDGE_TAIL = 2304, 8  # bytes of the next / previous block a rank's own kernels may read: the last tile of 2048
                                # positions + 64 symbols of look-ahead past the block's end; the byte before its start
HIST_SAMPLE_MIN = 1 << 24      # blocks of at least this many positions take their cut points from a sampled histogram
HIST_SAMPLE_STRIDE = 8         # ... of every 8th tile of 2048 positions


def bwt_slice(text: torch.Tensor, sa_slice: torch.Tensor) -> torch.Tensor:
    out = _empty(sa_slice.numel(), torch.uint8, text.device)
    fn = _lib.load().hkcsa_bwt_slice64 if sa_slice.dtype == torch.int64 else _lib.load().hkcsa_bwt_slice
    check(fn(_ptr(text), text.numel(), _ptr(sa_slice), sa_slice.numel(), _ptr(out), _stream()))
    return out


@dataclass
class SuffixArraySlice:
    rank: int
    world: int
    n: int                      # length of the whole text
    offset: int                 # global SA position of this slice's first entry
    sa: torch.Tensor            # sorted suffix ids: uint32 bit patterns in int32 storage, or int64 (wide)
    bwt: torch.Tensor           # uint8, same length
    text: torch.Tensor          # the replicated text
    bucket_range: tuple
    rounds: list = field(default_factory=list)        # working-set size per refinement round (this rank)
    ext_rounds: int = 0
    dbl_rounds: int = 0
    phases: dict = field(default_factory=dict)        # seconds per phase (profile=True)
    nvlink_bytes_in: int = 0                          # bytes this GPU received: text blocks + (key, id) pairs

    def sa_int64(self) -> torch.Tensor:
        return self.sa if self.sa.dtype == torch.int64 else self.sa.to(torch.int64) & 0xFFFFFFFF


def _u64arr(vals):
    return (C.c_uint64 * len(vals))(*[int(v) for v in vals])


def _align(x: int, a: int = 256) -> int:
    return (x + a - 1) // a * a


def _rank_program(rank: int, world: int, block: torch.Tensor, wide, profile: bool, ext_rounds_max: int,
                  group_round: bool = True, hist_stride: int | None = None):
    """One rank's build as a generator.  Yields ("gather", array) -> [world, len] int64 numpy; ("text_async", block,
    sizes) -> (the text buffer with this rank's block and its edges in place, start and wait functions for the rest);
    ("symm", nbytes) -> (uint8 tensor, [address of every rank's buffer]); ("barrier",)."""
    L = _lib.load()
    dev = block.device
    phases: dict = {}
    t_last = [0.0]

    def tick(name=None):
        if not profile:
            return
        torch.cuda.synchronize(dev)
        now = time.perf_counter()
        if name is not None:
            phases[name] = phases.get(name, 0.0) + now - t_last[0]
        t_last[0] = now

    tick()
    # ---- 1. the text on every rank
    sizes = (yield ("gather", np.array([block.numel()], dtype=np.int64)))[:, 0]
    n = int(sizes.sum())
    if n > (1 << 40):
        raise _lib.HkcsaError(_lib.ERANGE, f"text of {n} symbols exceeds 2^40")
    starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    # The blocks travel while this rank already works on its own: histograms, cut points and the bucket exchange read
    # the rank's own block only (+ the first bytes of the next block for the keys at its end and the last byte of the
    # block before it), the whole text is first needed by the refinement rounds -- text_ready() makes the stream wait.
    # text_start() launches the collective: at once.  HKCSA_DSA_TEXT_LATE=1 holds it back until the bucket exchange is
    # over, so that the two do not share the NVLink ingress -- measured on 4 GPUs x 1 GB: the exchange is no faster
    # (15.9 ms either way: the packing bounds it), the round-0 sort beside the collective is slower (55.6 against 54.0 ms).
    text, text_start, text_ready = yield ("text_async", block, sizes)
    if os.environ.get("HKCSA_DSA_TEXT_LATE") != "1":
        text_start()
    begin, end = int(starts[rank]), int(starts[rank + 1])
    tick("text_allgather")
    # ---- 2. one prefix code and one set of cut points for everybody
    bh = (yield ("gather", byte_hist(block).astype(np.int64))).sum(0).astype(np.uint64)
    plan = DsaPlan()
    check(L.hkcsa_dsa_plan_make(bh.ctypes.data_as(C.POINTER(C.c_uint64)), n, 1 if wide else 0, C.byref(plan)))
    is_wide = bool(plan.wide)
    d_hist = torch.empty(_lib.DSA_BUCKETS, dtype=torch.int64, device=dev)
    # the exact bucket histogram costs one global atomic per suffix; big blocks histogram a sample of their tiles for
    # the cut points and count their suffixes per owner under those cuts in a second, atomics-free pass (the regions
    # of the exchange must be sized exactly)
    stride = hist_stride if hist_stride is not None else (HIST_SAMPLE_STRIDE if int(sizes.max()) >= HIST_SAMPLE_MIN else 1)
    if stride > 1:
        check(L.hkcsa_dsa_bucket_hist_sampled(_ptr(text), C.byref(plan), begin, end, stride, _ptr(d_hist), _stream()))
        hist_all = yield ("gather", d_hist)
        ranges = balanced_bucket_ranges(np.asarray(hist_all, dtype=np.int64).sum(0), world)
        cuts0 = [r[0] for r in ranges] + [_lib.DSA_BUCKETS]
        d_cnt = torch.empty(_lib.DSA_MAX_RANKS, dtype=torch.int64, device=dev)
        check(L.hkcsa_dsa_dest_counts(_ptr(text), C.byref(plan), begin, end, world,
                                      (C.c_uint32 * (world + 1))(*[int(c) for c in cuts0]), _ptr(d_cnt), _stream()))
        cnt_all = (yield ("gather", d_cnt))[:, :world]
        cuts, cnt, counts, slice_off = exchange_layout_from_counts(cuts0, cnt_all)
    else:
        check(L.hkcsa_dsa_bucket_hist(_ptr(text), C.byref(plan), begin, end, _ptr(d_hist), _stream()))
        hist_all = yield ("gather", d_hist)
        cuts, cnt, counts, slice_off = exchange_layout(hist_all, world)
    if int(counts.max()) > _lib.MAX_N:
        raise _lib.HkcsaError(_lib.ERANGE, f"a slice of {int(counts.max())} suffixes exceeds {_lib.MAX_N}: the buckets "
                                           "(top 16 key bits) of this text are too uneven for this many ranks")
    M = int(counts[rank])
    cap = _align(max(int(counts.max()), 1), 64)
    tick("histograms")
    # ---- 3. symmetric workspace: receive arrays + ISA block, the same layout on every rank
    id_bytes = 8 if is_wide else 4
    blk = max(1, -(-n // world))                                # positions per ISA block
    off_keys = 0
    off_va = _align(off_keys + 8 * cap)
    off_vb = _align(off_va + 4 * cap)
    off_ids64 = _align(off_vb + 4 * cap)
    off_isa = _align(off_ids64 + (8 * cap if is_wide else 0))
    total = _align(off_isa + id_bytes * blk)
    ws, ptrs = yield ("symm", total)
    keys = ws[off_keys:off_keys + 8 * cap].view(torch.int64)
    val_a = ws[off_va:off_va + 4 * cap].view(torch.int32)
    val_b = ws[off_vb:off_vb + 4 * cap].view(torch.int32)
    ids64 = ws[off_ids64:off_ids64 + 8 * cap].view(torch.int64) if is_wide else None
    isa = ws[off_isa:off_isa + id_bytes * blk]
    off_ids = off_ids64 if is_wide else off_va
    yield ("barrier",)                                          # nobody still reads the workspace of an earlier build
    tick("workspace")
    # ---- 4. pack + partition + exchange in one kernel
    d_counters = torch.empty(_lib.DSA_MAX_RANKS, dtype=torch.int64, device=dev)
    h_cuts = (C.c_uint32 * (world + 1))(*[int(c) for c in cuts])
    base = [int(cnt[:rank, d].sum()) for d in range(world)]
    check(L.hkcsa_dsa_pack_exchange(_ptr(text), C.byref(plan), begin, end, world, h_cuts,
                                    _u64arr([p + off_keys for p in ptrs]), _u64arr([p + off_ids for p in ptrs]),
                                    _u64arr(base), _ptr(d_counters), _stream()))
    yield ("barrier",)                                          # every pair has landed
    tick("pack_exchange")
    text_start()
    # ---- 5. local sort + refinement
    state = C.create_string_buffer(L.hkcsa_dsa_state_bytes())
    nscratch = L.hkcsa_dsa_scratch_bytes(cap)
    scratch = _scratch(nscratch, dev)
    check(L.hkcsa_dsa_begin(state, C.byref(plan), _ptr(text), _ptr(keys), _ptr(ids64) if is_wide else _ptr(val_a),
                            _ptr(val_a), _ptr(val_b), M, cap, _ptr(scratch), nscratch, _stream()))
    tick("sort_round0")
    text_ready()
    tick("text_wait")
    slice_ptr = L.hkcsa_dsa_slice(state) or (val_a.data_ptr())
    off_slice = off_va if slice_ptr == val_a.data_ptr() else off_vb
    ext_done, dbl_done, prev_all = 0, 0, None
    isa_ready = False
    group_round_due = group_round
    peer_isa = _u64arr([p + off_isa for p in ptrs])
    peer_sa = _u64arr([p + off_slice for p in ptrs])
    peer_ids64 = _u64arr([p + off_ids64 for p in ptrs]) if is_wide else None
    h_slice_off = _u64arr(slice_off)
    while True:
        m_all = int((yield ("gather", np.array([L.hkcsa_dsa_working_set(state)], dtype=np.int64))).sum())
        if m_all == 0:
            break
        if group_round_due:
            # first: every small group ordered by direct text comparison, no radix sort, no communication -- after
            # round 0 nearly all groups hold two or three suffixes.  Skipped for repetitive texts (most suffixes tied).
            group_round_due = False
            if 2 * m_all <= n:
                check(L.hkcsa_dsa_group_round(state, _stream()))
                tick("group_round")
                continue
        stalled = prev_all is not None and ext_done >= 2 and 2 * m_all > prev_all
        prev_all = m_all
        if not isa_ready and ext_done < ext_rounds_max and not stalled:
            check(L.hkcsa_dsa_ext_round(state, _stream()))
            ext_done += 1
            tick("extension_rounds")
            continue
        if not isa_ready:                                       # switch to rank doubling: enter the working set
            isa.fill_(0xFF)
            yield ("barrier",)
            check(L.hkcsa_dsa_isa_publish(state, world, peer_isa, blk, int(slice_off[rank]), 0, _stream()))
            yield ("barrier",)
            isa_ready = True
        check(L.hkcsa_dsa_dbl_keys(state, world, peer_isa, blk, peer_sa, peer_ids64, h_slice_off, h_cuts, _stream()))
        yield ("barrier",)                                      # every rank has read the ranks of this generation
        check(L.hkcsa_dsa_dbl_sort(state, _stream()))
        check(L.hkcsa_dsa_isa_publish(state, world, peer_isa, blk, int(slice_off[rank]), 1, _stream()))
        yield ("barrier",)
        dbl_done += 1
        tick("doubling_rounds")
    # ---- 6. the slice leaves the workspace; BWT of the slice
    if is_wide:                     # ids and BWT symbols arrive together (the symbol rides in the id's top byte)
        sa = _empty(M, torch.int64, dev)
        bw = _empty(M, torch.uint8, dev)
        check(L.hkcsa_dsa_gather_ids64(state, _ptr(sa), _ptr(bw), _stream()))
    else:
        sa = (val_a if off_slice == off_va else val_b)[:M].clone()
        bw = bwt_slice(text, sa)
    sent = int(d_counters.cpu().numpy()[:world].sum())
    if sent != end - begin:
        raise RuntimeError(f"exchange sent {sent} pairs for a block of {end - begin} positions")
    yield ("barrier",)                                          # peers may have been searching this rank's slice
    tick("slice_and_bwt")
    nr = C.c_uint32(0)
    elems = (C.c_uint64 * 48)()
    check(L.hkcsa_dsa_rounds(state, C.byref(nr), elems, 48))
    received = (n - (end - begin)) + (M - int(cnt[rank, rank])) * (8 + id_bytes)
    return SuffixArraySlice(rank, world, n, int(slice_off[rank]), sa, bw, text, (int(cuts[rank]), int(cuts[rank + 1])),
                            [int(elems[r]) for r in range(min(int(nr.value), 48))], ext_done, dbl_done, phases, received)


# ------------------------------------------------------------------ running the program: torch.distributed
_WORKSPACES: dict = {}


class _SymmWorkspace:
    """One symmetric-memory allocation per process group, grown on demand and reused by later builds (allocating
    and mapping gigabytes of peer memory costs far more than the build itself)."""

    def __init__(self, nbytes: int, device, group):
        import torch.distributed._symmetric_memory as symm
        self.nbytes = int(nbytes)
        self.buf = symm.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.hdl = symm.rendezvous(self.buf, group)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]


def _all_gather_rows(t: torch.Tensor, world: int, group) -> torch.Tensor:
    """[world, len] from one row per rank: one collective (NCCL), or the list form for gloo (CPU tests)."""
    import torch.distributed as dist
    t = t.contiguous()
    if t.is_cuda:
        out = torch.empty((world, t.numel()), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t, group=group)
        return out
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t, group=group)
    return torch.stack(parts)


_SIDE_GROUPS: dict = {}


def _side_group(group):
    """A second communicator over the same ranks, for the text all-gather that runs beside the build: collectives of
    one communicator execute in order, so the small all-gathers of the build (histograms, counts) would queue up
    behind the text on the main one.  Created once per group (collectively: every rank gets here in the same order)."""
    import torch.distributed as dist
    key = id(group) if group is not None else 0
    if key not in _SIDE_GROUPS:
        ranks = dist.get_process_group_ranks(group if group is not None else dist.group.WORLD)
        _SIDE_GROUPS[key] = dist.new_group(ranks=ranks)
    return _SIDE_GROUPS[key]


def _torch_run(prog, group, device):
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    ws = None
    try:
        req = next(prog)
        while True:
            kind = req[0]
            if kind == "gather":
                x = req[1]
                t = x.to(torch.int64) if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.int64)).to(device)
                res = _all_gather_rows(t, world, group).cpu().numpy()
            elif kind == "text_async":
                block, sizes = req[1], [int(v) for v in req[2]]
                if len(set(sizes)) == 1 and sizes[0] >= EDGE_HEAD + EDGE_TAIL and hasattr(dist, "all_gather_into_tensor"):
                    # equal blocks: ONE in-place all-gather into the text buffer, left running on NCCL's stream.  The
                    # edges (first bytes / last bytes of every block) go ahead in a small collective of their own.
                    m = sizes[0]
                    text = torch.empty(m * world, dtype=torch.uint8, device=device)
                    own = text[rank * m:(rank + 1) * m]
                    own.copy_(block)
                    edges = _all_gather_rows(torch.cat([block[:EDGE_HEAD], block[m - EDGE_TAIL:]]), world, group)
                    if rank + 1 < world:
                        text[(rank + 1) * m:(rank + 1) * m + EDGE_HEAD] = edges[rank + 1, :EDGE_HEAD]
                    if rank > 0:
                        text[rank * m - EDGE_TAIL:rank * m] = edges[rank - 1, EDGE_HEAD:]
                    pending = []

                    def start(text=text, own=own, pending=pending):     # idempotent: the program may call it twice
                        if not pending:
                            pending.append(dist.all_gather_into_tensor(text, own, group=_side_group(group), async_op=True))

                    def wait(pending=pending, start=start):
                        start()
                        pending[0].wait()

                    res = (text, start, wait)
                else:                                           # one collective on padded blocks, then compaction
                    width = max(sizes)
                    pad = torch.zeros(width, dtype=torch.uint8, device=device)
                    pad[: block.numel()] = block
                    allb = _all_gather_rows(pad, world, group)
                    res = (torch.cat([allb[r, : sizes[r]] for r in range(world)]), lambda: None, lambda: None)
            elif kind == "symm":
                need = torch.tensor([int(req[1])], dtype=torch.int64, device=device)
                dist.all_reduce(need, op=dist.ReduceOp.MAX, group=group)
                need = int(need.item())
                key = (id(group) if group is not None else 0, torch.device(device).index)
                ws = _WORKSPACES.get(key)
                if ws is None or ws.nbytes < need:
                    _WORKSPACES.pop(key, None)
                    ws = _SymmWorkspace(need + need // 8, device, group if group is not None else dist.group.WORLD)
                    _WORKSPACES[key] = ws
                res = (ws.buf, ws.ptrs)
            elif kind == "barrier":
                if ws is not None:
                    ws.hdl.barrier()                            # device-side, on the current stream
                else:
                    dist.barrier(group=group)
                res = None
            else:
                raise ValueError(kind)
            req = prog.send(res)
    except StopIteration as done:
        return done.value


def distributed_suffix_array(local_block: torch.Tensor, group=None, wide: bool | None = None, profile: bool = False,
                             ext_rounds_max: int = EXT_ROUNDS_MAX, group_round: bool = True,
                             hist_stride: int | None = None) -> SuffixArraySlice:
    """local_block: this rank's contiguous part of the text (uint8, on this rank's GPU), blocks in rank order.
    Collective: every rank of `group` calls it.  profile=True synchronises at phase boundaries and fills
    SuffixArraySlice.phases."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    if world > _lib.DSA_MAX_RANKS:
        raise ValueError(f"at most {_lib.DSA_MAX_RANKS} ranks")
    prog = _rank_program(dist.get_rank(group), world, local_block, wide, profile, ext_rounds_max, group_round, hist_stride)
    return _torch_run(prog, group, local_block.device)


def release_workspaces() -> None:
    _WORKSPACES.clear()


# ------------------------------------------------------------------ running the program: ranks emulated on one GPU
def emulate_distributed_suffix_array(blocks, wide: bool | None = None, ext_rounds_max: int = EXT_ROUNDS_MAX,
                                     profile: bool = False, group_round: bool = True, hist_stride: int | None = None):
    """The same per-rank programs, advanced in lockstep inside one process: `blocks` are the ranks' text blocks on
    ONE GPU, peers' buffers are plain device buffers of the same process.  Returns the slices in rank order."""
    world = len(blocks)
    if not 1 <= world <= _lib.DSA_MAX_RANKS:
        raise ValueError(f"1..{_lib.DSA_MAX_RANKS} ranks")
    dev = blocks[0].device
    progs = [_rank_program(r, world, blocks[r], wide, profile, ext_rounds_max, group_round, hist_stride) for r in range(world)]
    reqs = [next(p) for p in progs]
    results = [None] * world
    live = list(range(world))
    while live:
        kind = reqs[live[0]][0]
        assert all(reqs[r][0] == kind for r in live), "rank programs diverged"
        if kind == "gather":
            rows = [reqs[r][1].cpu().numpy() if isinstance(reqs[r][1], torch.Tensor) else np.asarray(reqs[r][1])
                    for r in live]
            res = [np.stack(rows).astype(np.int64)] * world
        elif kind == "text_async":
            full = torch.cat([reqs[r][1] for r in live])
            res = [(full, lambda: None, lambda: None)] * world
        elif kind == "symm":
            need = max(int(reqs[r][1]) for r in live)
            bufs = [torch.empty(need, dtype=torch.uint8, device=dev) for _ in live]
            ptrs = [b.data_ptr() for b in bufs]
            res = [(bufs[r], ptrs) for r in range(world)]
        elif kind == "barrier":
            res = [None] * world                                # one stream: program order is the barrier
        else:
            raise ValueError(kind)
        nxt = []
        for r in live:
            try:
                reqs[r] = progs[r].send(res[r])
                nxt.append(r)
            except StopIteration as done:
                results[r] = done.value
        assert not nxt or len(nxt) == len(live), "rank programs must finish together"
        live = nxt
    return results


# ------------------------------------------------------------------ queries over a sliced index
class MultiSliceIndex:
    """FM index over a BWT that exists as slices (one per rank of the distributed build).  Every slice has its
    own wavelet tree and sampled SA; occ(c, i) = occurrences in earlier slices + a rank walk inside the slice
    holding row i (csrc/multi_slice.cu).  All slices are resident on this GPU (they are all-gathered after the
    build), so count / locate run locally and the pattern batch can be sharded exactly as for one index."""

    def __init__(self, n: int, slices, sa_sample_rate: int = 0):
        """slices: list of dicts with 'bwt' (uint8 tensor) and, for locate, 'sa' (uint32-as-int32 or int64 tensor),
        in rank order.  Builds the per-slice structures with libhkcsa K3 / the sampled-SA kernels."""
        from .engine import DeviceWaveletTree
        self.n = n
        self.device = slices[0]["bwt"].device
        self.wts, self.ssas = [], []
        self.row0 = -1
        starts = [0]
        for sl in slices:
            bw = sl["bwt"]
            self.wts.append(DeviceWaveletTree(bw))
            if sa_sample_rate > 0:
                self.ssas.append(_sampled_sa_slice(sl["sa"], sa_sample_rate))
                hit = (sl["sa"] == 0).nonzero()                   # plumbing: where suffix 0 is
                if hit.numel():
                    self.row0 = starts[-1] + int(hit[0, 0])
            starts.append(starts[-1] + bw.numel())
        if starts[-1] != n:
            raise ValueError("slice lengths do not add up to n")
        self.starts = starts
        self.rate = sa_sample_rate
        self._assemble()

    @classmethod
    def from_parts(cls, n, starts, wt_parts, ssa_parts, rate, row0):
        """wt_parts: [(WtPlan, blob tensor)], ssa_parts: [(SsaPlan, blob tensor)] or [] -- replicas.  row0: the
        global row of suffix 0 (-1 without ssa_parts); the exact LF step of locate needs it."""
        from .engine import DeviceWaveletTree, SampledSA
        self = cls.__new__(cls)
        self.n, self.starts, self.rate, self.row0 = n, list(starts), rate, int(row0)
        self.device = wt_parts[0][1].device
        self.wts = []
        for plan, blob in wt_parts:
            wt = DeviceWaveletTree.__new__(DeviceWaveletTree)
            wt.device, wt.n, wt.hist, wt.plan, wt.blob = blob.device, int(plan.n), None, plan, blob
            self.wts.append(wt)
        self.ssas = [SampledSA(p, b) for p, b in ssa_parts]
        self._assemble()
        return self

    def _assemble(self):
        L = _lib.load()
        S = len(self.wts)
        if not 1 <= S <= _lib.MAX_SLICES:
            raise ValueError(f"1..{_lib.MAX_SLICES} slices")
        self.desc = torch.zeros(L.hkcsa_multi_desc_bytes(), dtype=torch.uint8, device=self.device)
        blobs = (C.c_void_p * S)(*[w.blob.data_ptr() for w in self.wts])
        plans = (C.POINTER(_lib.WtPlan) * S)(*[C.pointer(w.plan) for w in self.wts])
        starts = (C.c_uint64 * (S + 1))(*self.starts)
        if self.ssas:
            sblobs = (C.c_void_p * S)(*[s.blob.data_ptr() for s in self.ssas])
            splans = (C.POINTER(_lib.SsaPlan) * S)(*[C.pointer(s.plan) for s in self.ssas])
        else:
            sblobs, splans = None, None
        row0 = self.row0 if self.row0 >= 0 else (1 << 64) - 1
        check(L.hkcsa_multi_desc_build(S, blobs, plans, starts, sblobs, splans, row0, _ptr(self.desc), _stream()))

    def count_batch(self, pat: torch.Tensor, off: torch.Tensor):
        P = off.numel() - 1
        lo = _empty(P, torch.int64, self.device)
        hi = _empty(P, torch.int64, self.device)
        check(_lib.load().hkcsa_multi_count_batch(_ptr(self.desc), _ptr(pat), _ptr(off), P, _ptr(lo), _ptr(hi), _stream()))
        return lo, hi

    def locate_batch(self, pat: torch.Tensor, off: torch.Tensor):
        """CSR (offsets int64[P+1], positions int64 in SA order) through LF walks across slices."""
        if not self.ssas:
            raise ValueError("index was built without a sampled suffix array")
        out_off, rows = _expand_ranges(*self.count_batch(pat, off), wide=True)
        return out_off, self.locate_rows(rows)

    def locate_rows(self, rows: torch.Tensor) -> torch.Tensor:
        """int64 global rows -> int64 text positions (SA[row]) through LF walks across slices; -1 only for a walk
        over a corrupt index."""
        if not self.ssas:
            raise ValueError("index was built without a sampled suffix array")
        rows = rows.to(device=self.device, dtype=torch.int64).contiguous()
        out = _empty(rows.numel(), torch.int64, self.device)
        check(_lib.load().hkcsa_multi_locate_rows(_ptr(self.desc), _ptr(rows), rows.numel(), _ptr(out), _stream()))
        return out

    # extract (csrc/extract.cu): text[begin:end) from the slices alone, with the exact LF step on every text
    def isa_samples(self) -> torch.Tensor:
        """int64[S + 1]: the global row of the suffix at text position k * rate for k < S = ceil(n / rate), and
        [S] = [0].  Derived from the slices' sampled suffix arrays; built on first use."""
        if not self.ssas:
            raise ValueError("index was built without a sampled suffix array")
        if getattr(self, "_isa", None) is None:
            S = len(self.ssas)
            out = _empty(-(-self.n // self.rate) + 1, torch.int64, self.device)
            blobs = (C.c_void_p * S)(*[s.blob.data_ptr() for s in self.ssas])
            plans = (C.POINTER(_lib.SsaPlan) * S)(*[C.pointer(s.plan) for s in self.ssas])
            starts = (C.c_uint64 * (S + 1))(*self.starts)
            check(_lib.load().hkcsa_multi_isa_samples(S, blobs, plans, starts, _ptr(out), _stream()))
            self._isa = out
        return self._isa

    def extract_batch(self, begin: torch.Tensor, end: torch.Tensor):
        """text[begin[q]:end[q]) for every q (int64 tensors; 0 <= begin <= end <= n, sentinel included) ->
        (out_off int64[R+1], bytes uint8[total]) on the device, request q at bytes[out_off[q]:out_off[q+1]]."""
        if not self.ssas:
            raise ValueError("index was built without a sampled suffix array")
        L = _lib.load()
        begin, end, out_off, out = _extract_requests(begin, end, self.n, self.device)
        if out.numel() == 0:
            return out_off, out
        R = begin.numel()
        isa = self.isa_samples()
        nbytes = L.hkcsa_extract_scratch_bytes(R)
        scratch = _scratch(nbytes, self.device)
        check(L.hkcsa_multi_extract(_ptr(self.desc), self.n, self.rate, _ptr(isa), _ptr(begin), _ptr(end),
                                    _ptr(out_off), R, _ptr(out), _ptr(scratch), nbytes, _stream()))
        return out_off, out

    def extract(self, begin: int, end: int) -> torch.Tensor:
        """text[begin:end) of the indexed text (sentinel included) as a uint8 device tensor."""
        b = torch.tensor([begin], dtype=torch.int64, device=self.device)
        e = torch.tensor([end], dtype=torch.int64, device=self.device)
        return self.extract_batch(b, e)[1]


def _sampled_sa_slice(sa_slice: torch.Tensor, rate: int):
    """Marks + samples for the rows of one slice (suffix ids are global, uint32 bit patterns)."""
    from .engine import SampledSA
    L = _lib.load()
    m = sa_slice.numel()
    wide = sa_slice.dtype == torch.int64
    ids = sa_slice if wide else (sa_slice.to(torch.int64) & 0xFFFFFFFF)
    n_marks = int((ids % rate == 0).sum().item())            # plumbing: sizes the sample array
    plan = _lib.SsaPlan()
    check(L.hkcsa_ssa_plan_make_slice(m, rate, n_marks, C.byref(plan)))
    blob = torch.zeros(int(plan.blob_bytes), dtype=torch.uint8, device=sa_slice.device)
    scratch = _scratch(plan.scratch_bytes, sa_slice.device)
    fn = L.hkcsa_ssa_build64 if wide else L.hkcsa_ssa_build
    check(fn(_ptr(sa_slice), C.byref(plan), _ptr(blob), _ptr(scratch), int(plan.scratch_bytes), _stream()))
    return SampledSA(plan, blob)


def replicate_sliced_index(sl: SuffixArraySlice, sa_sample_rate: int = 32, group=None) -> MultiSliceIndex:
    """After distributed_suffix_array: every rank builds the wavelet tree and sampled SA of ITS slice; the plan
    structs travel in one all-gather, the blobs (padded to the largest) in one all-gather each, and every rank
    assembles the same MultiSliceIndex over views of the gathered buffers."""
    import torch.distributed as dist
    from .engine import DeviceWaveletTree
    world, rank, dev = sl.world, sl.rank, sl.sa.device
    wt = DeviceWaveletTree(sl.bwt)
    ssa = _sampled_sa_slice(sl.sa, sa_sample_rate) if sa_sample_rate > 0 else None
    wsz, ssz = C.sizeof(_lib.WtPlan), C.sizeof(_lib.SsaPlan)
    mine0 = -1                                               # my global row of suffix 0, or -1
    if ssa is not None:
        hit = (sl.sa == 0).nonzero()
        mine0 = sl.offset + int(hit[0, 0]) if hit.numel() else -1
    H = 32
    head = torch.zeros(H + wsz + ssz, dtype=torch.uint8)
    head[:H] = torch.from_numpy(np.array([sl.sa.numel(), wt.blob.numel(), ssa.blob.numel() if ssa is not None else 0,
                                          mine0], dtype=np.int64).view(np.uint8))
    head[H:H + wsz] = torch.frombuffer(bytearray(bytes(wt.plan)), dtype=torch.uint8)
    if ssa is not None:
        head[H + wsz:] = torch.frombuffer(bytearray(bytes(ssa.plan)), dtype=torch.uint8)
    heads = torch.empty((world, head.numel()), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(heads, head.to(dev), group=group)
    heads = heads.cpu().numpy()
    meta = [heads[r, :H].view(np.int64).tolist() for r in range(world)]
    starts = [0]
    for r in range(world):
        starts.append(starts[-1] + meta[r][0])

    def gather_blobs(mine, sizes):
        width = (max(sizes) + 255) // 256 * 256              # rows stay 32-byte aligned (rank blocks)
        pad = torch.zeros(width, dtype=torch.uint8, device=dev)
        if mine is not None:
            pad[: mine.numel()] = mine
        allb = torch.empty((world, width), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allb, pad, group=group)
        return [allb[r, : sizes[r]] for r in range(world)]

    wt_blobs = gather_blobs(wt.blob, [m[1] for m in meta])
    wt_parts = [(_lib.WtPlan.from_buffer_copy(heads[r, H:H + wsz].tobytes()), wt_blobs[r]) for r in range(world)]
    ssa_parts = []
    if sa_sample_rate > 0:
        ssa_blobs = gather_blobs(ssa.blob, [m[2] for m in meta])
        ssa_parts = [(_lib.SsaPlan.from_buffer_copy(heads[r, H + wsz:].tobytes()), ssa_blobs[r]) for r in range(world)]
    row0 = max(m[3] for m in meta)
    return MultiSliceIndex.from_parts(sl.n, starts, wt_parts, ssa_parts, sa_sample_rate, row0)
