"""Plain torch references for the whole index, exact and independent of libhkcsa (no `hkcsa` import).

The CPU oracle sorts suffixes by comparison, which is too slow at n = 2^30 and on repetitive texts.  These functions
are linear or n log n, run on CPU tensors as well as CUDA tensors, and are pinned to the oracle on small inputs by
tests/test_device_reference.py.  Every function works in chunks: at n = 2^30 its peak beside its inputs stays within
about 16 GB (check_suffix_array: the int32 ISA + ~1 GB; symbol_positions: int32[n] + ~1 GB), except entropy_hk, whose
torch.unique over n packed int64 windows takes about 3 x 8 B x n (26 GB at 2^30).  Past 2^31 - 1 symbols (the
distributed build) rows and suffix ids no longer fit int32: the ISA and the row lists are int64 there (about 17 GB
+ ~1 GB each at 2^31), and `wide=True` forces that form at any size.  Suffix arrays may be int32 or int64.

Conventions are those of the package: suffixes compare as byte strings and a proper prefix sorts first; ranges are
inclusive (lo, hi) with (-1, -1) for a miss and (0, n-1) for the empty pattern; rank(p) counts ones in [0, p);
select(k) is the smallest p with rank(p) >= k.
"""
from __future__ import annotations

import torch

CHUNK = 1 << 24          # rows per chunk: a handful of int64[CHUNK] temporaries (128 MB each)


def _chunks(n: int, chunk: int = CHUNK):
    for a in range(0, n, chunk):
        yield a, min(n, a + chunk)


# ------------------------------------------------------------------ suffix array
INT32_MAX = (1 << 31) - 1


def _row_dtype(n: int, wide: bool | None) -> torch.dtype:
    """int32 while every row and suffix id < n fits it, else (or with wide=True) int64."""
    return torch.int64 if wide or n > INT32_MAX else torch.int32


def check_suffix_array(text: torch.Tensor, sa: torch.Tensor, chunk: int = CHUNK, *, wide: bool | None = None
                       ) -> torch.Tensor:
    """The O(n) checker of Burkhardt and Kaerkkaeinen.  `sa` is the suffix array of `text` iff it is a permutation of
    [0, n) and, with R[j] = ISA[j] for j < n and R[n] = -1, every row i has
        (text[sa[i]], R[sa[i] + 1]) < (text[sa[i+1]], R[sa[i+1] + 1])   (strictly).
    Raises AssertionError naming the first bad row; returns the ISA (int32[n], int64[n] past 2^31 - 1 or with
    wide=True)."""
    n = text.numel()
    assert sa.numel() == n, f"suffix array has {sa.numel()} entries for a text of {n}"
    dev = sa.device
    dt = _row_dtype(n, wide)
    if n == 0:
        return torch.empty(0, dtype=dt, device=dev)
    lo, hi = int(sa.min()), int(sa.max())
    assert 0 <= lo and hi < n, f"suffix array entries out of [0, {n}): min {lo}, max {hi}"
    isa = torch.empty(n, dtype=dt, device=dev)
    for a, b in _chunks(n, chunk):
        isa[sa[a:b].long()] = torch.arange(a, b, dtype=dt, device=dev)
    for a, b in _chunks(n, chunk):             # a duplicate leaves one of its rows overwritten by the other
        bad = isa[sa[a:b].long()] != torch.arange(a, b, dtype=dt, device=dev)
        if bool(bad.any()):
            i = a + int(bad.nonzero()[0, 0])
            raise AssertionError(f"suffix array is not a permutation: row {i} holds {int(sa[i])}, "
                                 f"which row {int(isa[int(sa[i])])} holds too")
    for a, b in _chunks(n - 1, chunk):        # pairs (a, a+1) ... (b-1, b)
        s = sa[a:b + 1].long()
        c = text[s].to(torch.int16)
        nxt = s + 1
        r = torch.where(nxt < n, isa[nxt.clamp(max=n - 1)].long(), torch.full_like(nxt, -1))
        bad = (c[:-1] > c[1:]) | ((c[:-1] == c[1:]) & (r[:-1] >= r[1:]))
        if bool(bad.any()):
            i = a + int(bad.nonzero()[0, 0])
            raise AssertionError(f"suffix array out of order at row {i}: suffixes {int(sa[i])} and {int(sa[i + 1])} "
                                 f"(first symbols {int(c[i - a])}, {int(c[i - a + 1])}; "
                                 f"ranks of their successors {int(r[i - a])}, {int(r[i - a + 1])})")
    return isa


def bwt_of(text: torch.Tensor, sa: torch.Tensor, chunk: int = CHUNK) -> torch.Tensor:
    """text[(sa - 1) mod n] (csa/bwt.py:3-13)."""
    n = text.numel()
    out = torch.empty(n, dtype=torch.uint8, device=text.device)
    for a, b in _chunks(n, chunk):
        out[a:b] = text[(sa[a:b].long() - 1) % n]
    return out


# ------------------------------------------------------------------ rank over the BWT
def symbol_positions(bwt: torch.Tensor, chunk: int = 1 << 25, *, wide: bool | None = None):
    """(pos int32[n], start int64[257]): the rows of every byte value in ascending order, values in byte order;
    the rows holding byte c are pos[start[c]:start[c+1]].  j = C[c] + occ(c, pos[j]) for every such row.  pos is
    int64 past 2^31 - 1 rows or with wide=True."""
    n = bwt.numel()
    dev = bwt.device
    cnt = torch.zeros(256, dtype=torch.int64, device=dev)
    for a, b in _chunks(n, chunk):
        cnt += torch.bincount(bwt[a:b].long(), minlength=256)
    start = torch.zeros(257, dtype=torch.int64, device=dev)
    start[1:] = torch.cumsum(cnt, 0)
    base = start[:256].clone()
    pos = torch.empty(n, dtype=_row_dtype(n, wide), device=dev)
    for a, b in _chunks(n, chunk):
        vals, order = torch.sort(bwt[a:b], stable=True)
        cc = torch.bincount(vals.long(), minlength=256)
        cstart = torch.cumsum(cc, 0) - cc
        v = vals.long()
        dest = base[v] + torch.arange(b - a, device=dev) - cstart[v]
        pos[dest] = (order + a).to(pos.dtype)
        base += cc
    return pos, start


def _lower_bound(arr: torch.Tensor, lo: torch.Tensor, hi: torch.Tensor, key: torch.Tensor) -> torch.Tensor:
    """Per query, the first index in [lo, hi) with arr[index] >= key (arr ascending on every such range)."""
    lo, hi = lo.clone(), hi.clone()
    for _ in range(64):
        live = lo < hi
        if not bool(live.any()):
            break
        mid = (lo + hi) // 2
        v = arr[mid.clamp(max=max(arr.numel() - 1, 0))].long()
        go_right = live & (v < key)
        lo = torch.where(go_right, mid + 1, lo)
        hi = torch.where(live & ~go_right, mid, hi)
    return lo


def occ_at(bwt: torch.Tensor, sym: torch.Tensor, pos: torch.Tensor, groups=None) -> torch.Tensor:
    """occ(sym[q], pos[q]): occurrences of byte sym[q] in bwt[0:pos[q]] (int64).  groups: symbol_positions(bwt), to
    reuse across calls."""
    p, start = groups if groups is not None else symbol_positions(bwt)
    c = sym.to(device=p.device).long()
    key = pos.to(device=p.device).long()
    return _lower_bound(p, start[c], start[c + 1], key) - start[c]


def bits_rank(bits: torch.Tensor, pos: torch.Tensor, chunk: int = 1 << 26) -> torch.Tensor:
    """Ones in bits[0:pos[q]] for 0 <= pos[q] <= len (int64): per chunk, a cumsum read at the requested positions."""
    n = bits.numel()
    pos = pos.to(device=bits.device).long()
    out = torch.zeros_like(pos)
    base = 0
    for a in range(0, n + 1, chunk):
        b = min(n, a + chunk)
        sel = (pos >= a) & (pos <= b) if b == n else (pos >= a) & (pos < b)
        idx = sel.nonzero().flatten()
        cs = torch.zeros(b - a + 1, dtype=torch.int64, device=bits.device)
        cs[1:] = torch.cumsum(bits[a:b], 0)
        out[idx] = base + cs[pos[idx] - a]
        base += int(cs[-1])
        if b == n:
            break
    return out


def bits_select(bits: torch.Tensor, k: torch.Tensor, chunk: int = 1 << 26) -> torch.Tensor:
    """For 1 <= k[q] <= ones: one past the position of the k-th one, i.e. the smallest p with rank(p) >= k (int64)."""
    n = bits.numel()
    k = k.to(device=bits.device).long()
    out = torch.full_like(k, -1)
    base = 0
    for a, b in _chunks(n, chunk):
        nz = bits[a:b].nonzero().flatten()
        sel = (k > base) & (k <= base + nz.numel())
        idx = sel.nonzero().flatten()
        out[idx] = a + nz[k[idx] - base - 1] + 1
        base += nz.numel()
    assert bool((out >= 0).all()), "select beyond the number of ones"
    return out


# ------------------------------------------------------------------ pattern ranges
def _windows(text: torch.Tensor, starts: torch.Tensor, m: int) -> torch.Tensor:
    """text[s : s+m] per start, past-the-end = -1 (sorts before every symbol) -> int16[Q, m]."""
    n = text.numel()
    idx = starts.long()[:, None] + torch.arange(m, device=text.device)
    w = text[idx.clamp(max=n - 1)].to(torch.int16)
    return torch.where(idx < n, w, torch.full_like(w, -1))


def _compare(text, sa, rows, pm, lens):
    """sign(suffix at row rows[q], truncated to lens[q] symbols - pattern q) in {-1, 0, 1}."""
    w = _windows(text, sa[rows].long(), pm.shape[1])
    live = torch.arange(pm.shape[1], device=pm.device)[None, :] < lens[:, None]
    diff = (w != pm) & live
    first = diff.to(torch.int8).argmax(1)
    d = (w.gather(1, first[:, None]) - pm.gather(1, first[:, None])).squeeze(1)
    return torch.where(diff.any(1), d.sign(), torch.zeros_like(d)).long()


def sa_range(text: torch.Tensor, sa: torch.Tensor, pats: torch.Tensor, off: torch.Tensor):
    """(lo, hi) int64[P] of every pattern pats[off[q]:off[q+1]] (m <= 64): the inclusive range of suffix-array rows
    whose suffixes start with it, by binary search over the (checked) suffix array; (-1, -1) for a miss, (0, n-1)
    for the empty pattern -- what find_range returns for every pattern that does not wrap around the text's end."""
    dev = sa.device
    n = text.numel()
    off = off.to(dev).long()
    P = off.numel() - 1
    lens = off[1:] - off[:-1]
    M = max(int(lens.max()) if P else 0, 1)
    assert M <= 64, "patterns of at most 64 symbols"
    j = torch.arange(M, device=dev)
    pidx = (off[:-1, None] + j).clamp(max=max(pats.numel() - 1, 0))
    pm = pats.to(dev)[pidx].to(torch.int16) if pats.numel() else torch.zeros(P, M, dtype=torch.int16, device=dev)
    pm = torch.where(j[None, :] < lens[:, None], pm, torch.zeros_like(pm))

    def bound(strict: bool):
        lo = torch.zeros(P, dtype=torch.int64, device=dev)
        hi = torch.full((P,), n, dtype=torch.int64, device=dev)
        while True:
            live = lo < hi
            if not bool(live.any()):
                return lo
            mid = (lo + hi) // 2
            c = _compare(text, sa, mid.clamp(max=n - 1), pm, lens)
            right = live & ((c <= 0) if strict else (c < 0))
            lo = torch.where(right, mid + 1, lo)
            hi = torch.where(live & ~right, mid, hi)

    first, past = bound(False), bound(True)
    hit = past > first
    neg = torch.full_like(first, -1)
    return torch.where(hit, first, neg), torch.where(hit, past - 1, neg)


# ------------------------------------------------------------------ H_k
def entropy_hk(text: torch.Tensor, k: int, chunk: int = CHUNK) -> float:
    """H_k in bits per symbol by the definition (DESIGN section 3): over the windows text[i:i+k+1], i < n-k, with c
    the count of a (k+1)-gram and T that of its k-symbol context, H_k = (sum T log2 T - sum c log2 c) / n, in fp64.
    0 for an empty text, k < 0, or n <= k.  Windows are packed into int64 at 8 bits per symbol for k <= 7, else at
    ceil(log2 sigma) bits per symbol (symbols replaced by their rank), e.g. k <= 20 on DNA + '$'."""
    n = text.numel()
    if n == 0 or k < 0 or (k > 0 and n <= k):
        return 0.0
    dev = text.device
    present = torch.bincount(text.long(), minlength=256) > 0
    sigma = int(present.sum())
    if (k + 1) * 8 <= 64:
        bits, code = 8, torch.arange(256, device=dev)
    else:
        bits = max(1, (sigma - 1).bit_length())
        if (k + 1) * bits > 64:
            raise ValueError(f"k = {k} windows over {sigma} symbols do not fit 64 bits")
        code = torch.cumsum(present.long(), 0) - 1
    W = n - k
    keys = torch.empty(W, dtype=torch.int64, device=dev)
    for a, b in _chunks(W, chunk):
        key = torch.zeros(b - a, dtype=torch.int64, device=dev)
        for t in range(k + 1):
            key = (key << bits) | code[text[a + t:b + t].long()]
        keys[a:b] = key
    grams, gcount = torch.unique(keys, sorted=True, return_counts=True)
    del keys
    # contexts are the top k symbols of a window: sorted grams keep every context contiguous
    ctx = grams >> bits if k > 0 else torch.zeros_like(grams)
    head = torch.ones_like(ctx, dtype=torch.bool)
    head[1:] = ctx[1:] != ctx[:-1]
    cid = torch.cumsum(head.long(), 0) - 1
    tcount = torch.zeros(int(cid[-1]) + 1, dtype=torch.int64, device=dev).index_add_(0, cid, gcount)

    def xlogx(c):
        c = c.double()
        return (c * torch.log2(c)).sum().item()

    return (xlogx(tcount) - xlogx(gcount)) / n


# ------------------------------------------------------------------ LF
def lf_invertible(bwt: torch.Tensor, isa: torch.Tensor, chunk: int = CHUNK) -> bool:
    """DESIGN section 3 K4c: LF inverts the suffix order iff row j0 = ISA[0] is the first row whose BWT symbol is
    bwt[j0]."""
    j0 = int(isa[0])
    c = bwt[j0]
    for a, b in _chunks(j0, chunk):
        if bool((bwt[a:b] == c).any()):
            return False
    return True
