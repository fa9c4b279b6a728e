"""Host-side engine over libhkcsa: device buffers, streams and the build / query
pipelines.  PyTorch is used for device memory, streams and (in dist.py)
torch.distributed only -- every computation is a libhkcsa kernel.

Pipeline (reference call stack, csa/enhanced_fm_index.py:8-13):
    text (+ '$') -> K1 suffix array -> K2 BWT -> byte histogram / C[] ->
    K3 wavelet tree + rank directories (replaces build_occ) [-> sampled SA]
Queries: K4 count (find_range), locate via the full SA (find) or via LF walks
to a sampled SA (CompressedSuffixArray.locate).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from ._lib import HkcsaError, OccPlan, RrrPlan, SaStats, SsaPlan, WtPlan, check

ENG96, DNA4 = 0, 1


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("hkcsa needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _ptr(t: torch.Tensor | None) -> int:
    return 0 if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _empty(n: int, dtype, device) -> torch.Tensor:
    return torch.empty(max(int(n), 0), dtype=dtype, device=device)


_STREAMS: dict = {}


def _aux_stream(device, which: str, priority: int = 0) -> "torch.cuda.Stream":
    """Long-lived side streams (one per device and purpose): the copy-out stream, the sampled-SA stream, and a
    high-priority stream for the critical path of the build's tail."""
    key = (torch.device(device).index, which)
    if key not in _STREAMS:
        _STREAMS[key] = torch.cuda.Stream(device=device, priority=priority)
    return _STREAMS[key]


def _scratch(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


class SymbolMap:
    """Order-preserving map between the code points of a ``str`` and bytes.

    The reference compares Python strings (csa/suffix_array.py:132), so any code point is a legal symbol.  Text in
    the latin-1 range maps to itself (one byte per code point, utils/data_loader.py:4).  A text with code points
    above 255 is re-coded: its distinct code points (plus those of `extra`, e.g. the '$' sentinel), sorted, become
    bytes 0, 1, 2, ... -- suffix order, BWT, C[] and every SA range are unchanged by an order-preserving re-coding.
    More than 256 distinct code points cannot be held in byte symbols: ValueError."""

    def __init__(self, text: str, extra: str = ""):
        self.back = None                      # identity
        self._cache = None                    # (text, its bytes): the constructor's probe is the encoding itself
        if text.isascii():                    # O(1) flag: nothing to probe, nothing to encode (see host_bytes)
            return
        try:
            self._cache = (text, text.encode("latin-1"))
        except UnicodeEncodeError:
            cps = sorted(set(text) | set(extra))
            if len(cps) > 256:
                raise ValueError(f"text holds {len(cps)} distinct symbols; byte symbols allow at most 256") from None
            self.back = cps
            self._fwd = {ord(c): i for i, c in enumerate(cps)}

    @classmethod
    def from_code_points(cls, back) -> "SymbolMap":
        """The map whose byte i is back[i] (an empty list: the identity map) -- what a saved index records."""
        self = cls.__new__(cls)
        self._cache = None
        self.back = list(back) or None
        if self.back is not None:
            self._fwd = {ord(c): i for i, c in enumerate(self.back)}
        return self

    @property
    def identity(self) -> bool:
        return self.back is None

    def encode(self, s: str):
        """bytes, or None when `s` holds a symbol outside the map (such a pattern cannot occur in the text)."""
        if self.back is None:
            if self._cache is not None and self._cache[0] is s:
                enc, self._cache = self._cache[1], None           # handed out once: do not pin 2x the text in memory
                return enc
            try:
                return s.encode("latin-1")
            except UnicodeEncodeError:
                return None
        if any(ord(c) not in self._fwd for c in set(s)):
            return None
        return s.translate(self._fwd).encode("latin-1")

    def host_bytes(self, s: str):
        """What to_device_u8 is given for the text `s`: the str itself when it is ASCII under the identity map (its own
        buffer is staged, no encoded copy), else encode(s)."""
        if self.back is None and s.isascii():
            return s
        return self.encode(s)

    def decode(self, b: bytes) -> str:
        if self.back is None:
            return b.decode("latin-1")
        return b.decode("latin-1").translate({i: c for i, c in enumerate(self.back)})

    def symbol(self, byte: int) -> str:
        return chr(byte) if self.back is None else self.back[byte]


_AsUTF8AndSize = C.pythonapi.PyUnicode_AsUTF8AndSize
_AsUTF8AndSize.restype = C.c_void_p
_AsUTF8AndSize.argtypes = [C.py_object, C.POINTER(C.c_ssize_t)]


def _staged_h2d(src, n: int, device, tail: bytes = b"") -> torch.Tensor:
    """n pageable host bytes at `src` (an address, or an object ctypes takes for one) + an optional tail (e.g. the
    sentinel) -> a fresh device tensor through hkcsa_h2d_staged: the library's pinned ring is filled by several host
    threads while the DMA of the chunks already staged runs on the current stream.  Returns once the source has been
    staged (it may be dropped); the copy completes in stream order."""
    out = torch.empty(n + len(tail), dtype=torch.uint8, device=device)
    L = _lib.load()
    with torch.cuda.device(out.device):
        if tail:                                           # first: its slot is long free when the bulk wants it
            check(L.hkcsa_h2d_staged(out.data_ptr() + n, tail, len(tail), 1, _stream()))
        if n:
            check(L.hkcsa_h2d_staged(out.data_ptr(), src, n, 0, _stream()))
    return out


def to_device_u8(data, device=None, tail: bytes = b"") -> torch.Tensor:
    """str (latin-1: utils/data_loader.py:4) / bytes / numpy / tensor -> contiguous uint8 CUDA tensor (`tail`
    appended: the callers that add the '$' sentinel do not build a second host copy for it).  An ASCII str is staged
    straight out of its own buffer (CPython keeps it at one byte per code point): no encoded copy is made."""
    device = device or _require_cuda()
    if isinstance(data, torch.Tensor):
        if data.dtype != torch.uint8:
            raise TypeError("text tensors must be uint8")
        d = data.to(device).contiguous()
        if tail:
            d = torch.cat([d, torch.tensor(list(tail), dtype=torch.uint8, device=d.device)])
        return d
    if isinstance(data, str):
        if data.isascii():
            if len(data) + len(tail) == 0:
                return torch.empty(0, dtype=torch.uint8, device=device)
            size = C.c_ssize_t(0)
            return _staged_h2d(_AsUTF8AndSize(data, C.byref(size)), len(data), device, tail)   # `data` outlives the call
        try:
            data = data.encode("latin-1")
        except UnicodeEncodeError:
            raise ValueError("text has code points above 255: encode it through engine.SymbolMap") from None
    if isinstance(data, (bytes, bytearray, memoryview)):
        arr = np.frombuffer(data, dtype=np.uint8)
    else:
        arr = np.ascontiguousarray(data, dtype=np.uint8)
    if arr.size + len(tail) == 0:
        return torch.empty(0, dtype=torch.uint8, device=device)
    return _staged_h2d(arr.ctypes.data, arr.size, device, tail)


_NP_OF = {torch.uint8: np.uint8, torch.int8: np.int8, torch.int16: np.int16, torch.int32: np.int32,
          torch.int64: np.int64, torch.float32: np.float32, torch.float64: np.float64}
TO_HOST_STAGED_MIN = 8 << 20


def to_host(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> numpy array in pageable memory.  From 8 MB on through hkcsa_d2h_staged (the pinned ring is
    drained by several host threads while the next chunks' DMAs run); below that torch's own copy."""
    nbytes = t.numel() * t.element_size()
    if not t.is_cuda or nbytes < TO_HOST_STAGED_MIN or t.dtype not in _NP_OF:
        return t.cpu().numpy()
    t = t.contiguous()
    out = np.empty(tuple(t.shape), dtype=_NP_OF[t.dtype])
    with torch.cuda.device(t.device):
        check(_lib.load().hkcsa_d2h_staged(out.ctypes.data, t.data_ptr(), nbytes, 0, _stream()))
    return out


# ------------------------------------------------------------------ workload
def gen_text(kind: int, seed: int, n: int, device=None) -> torch.Tensor:
    device = device or _require_cuda()
    out = _empty(n, torch.uint8, device)
    check(_lib.load().hkcsa_gen_text(kind, seed, n, _ptr(out), _stream()))
    return out


def gen_patterns(seed: int, P: int, text: torch.Tensor, alphabet: torch.Tensor, min_len: int = 8, max_len: int = 64):
    """Seeded substring patterns (half with one substitution): (bytes uint8[sum m], offsets int64[P+1])."""
    L = _lib.load()
    dev = text.device
    n = text.numel()
    lens = _empty(P, torch.int32, dev)
    check(L.hkcsa_gen_pattern_lengths(seed, P, min_len, max_len, n, _ptr(lens), _stream()))
    off = torch.zeros(P + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(lens, 0, dtype=torch.int64)   # plumbing: CSR offsets
    total = int(off[-1].item()) if P else 0
    out = _empty(total, torch.uint8, dev)
    check(L.hkcsa_gen_pattern_bytes(seed, P, _ptr(text), n, _ptr(alphabet), alphabet.numel(), _ptr(off), _ptr(out),
                                    _stream()))
    return out, off


# ------------------------------------------------------------------ K1 / K2
def suffix_array(text: torch.Tensor, stats: SaStats | None = None) -> torch.Tensor:
    """build_suffix_array (csa/suffix_array.py:131-134) on a device uint8 tensor -> int32[n]."""
    L = _lib.load()
    n = text.numel()
    if n > _lib.MAX_N:
        raise HkcsaError(_lib.ERANGE, f"text of {n} symbols exceeds the single-GPU limit {_lib.MAX_N}")
    sa = _empty(n, torch.int32, text.device)
    if n == 0:
        return sa
    nbytes = L.hkcsa_sa_scratch_bytes(n)
    scratch = _scratch(nbytes, text.device)
    st = stats if stats is not None else SaStats()
    check(L.hkcsa_sa_build(_ptr(text), n, _ptr(sa), _ptr(scratch), nbytes, _stream(), C.byref(st)))
    return sa


def suffix_array_bwt(text: torch.Tensor, stats: SaStats | None = None):
    """build_suffix_array + bwt_transform, the pair EnhancedFMIndex.__init__ runs (csa/enhanced_fm_index.py:10-11),
    in one call -> (int32[n], uint8[n]): with round-0 keys of at most 56 bits the BWT comes out of the sort."""
    L = _lib.load()
    n = text.numel()
    if n > _lib.MAX_N:
        raise HkcsaError(_lib.ERANGE, f"text of {n} symbols exceeds the single-GPU limit {_lib.MAX_N}")
    sa = _empty(n, torch.int32, text.device)
    out = _empty(n, torch.uint8, text.device)
    if n == 0:
        return sa, out
    nbytes = L.hkcsa_sa_scratch_bytes(n)
    scratch = _scratch(nbytes, text.device)
    st = stats if stats is not None else SaStats()
    check(L.hkcsa_sa_bwt_build(_ptr(text), n, _ptr(sa), _ptr(out), _ptr(scratch), nbytes, _stream(), C.byref(st)))
    return sa, out


def bwt(text: torch.Tensor, sa: torch.Tensor) -> torch.Tensor:
    """bwt_transform (csa/bwt.py:3-13) -> uint8[n]."""
    n = text.numel()
    if sa.numel() != n:
        raise IndexError("suffix array and text lengths differ")   # the reference would raise IndexError
    out = _empty(n, torch.uint8, text.device)
    check(_lib.load().hkcsa_bwt(_ptr(text), _ptr(sa), n, _ptr(out), _stream()))
    return out


def byte_hist(sym: torch.Tensor) -> np.ndarray:
    """Counts per byte value (host uint64[256]); the histogram under build_count (utils/utils.py:16-24)."""
    h = torch.empty(256, dtype=torch.int64, device=sym.device)
    check(_lib.load().hkcsa_byte_hist(_ptr(sym), sym.numel(), _ptr(h), _stream()))
    return h.cpu().numpy().astype(np.uint64)


def entropy_from_sa(text: torch.Tensor, sa: torch.Tensor, k: int) -> dict:
    """H_k of `text` (csa/high_order_entropy.py:4-32) from its suffix array, any k >= 0: one pass over the suffix
    array flags the runs of equal k- and (k+1)-grams.  Returns {"hk", "windows", "contexts", "grams"}."""
    n = text.numel()
    if n == 0 or k < 0:
        return {"hk": 0, "windows": 0, "contexts": 0, "grams": 0}
    if k == 0:
        hist = byte_hist(text).astype(np.float64)
        p = hist[hist > 0] / n
        return {"hk": float(-(p * np.log2(p)).sum()), "windows": n, "contexts": 1, "grams": int((hist > 0).sum())}
    if n <= k:
        return {"hk": 0, "windows": 0, "contexts": 0, "grams": 0}
    L = _lib.load()
    nbytes = L.hkcsa_entropy_scratch_bytes(n)
    scratch = _scratch(nbytes, text.device)
    out = (C.c_double * 5)()
    check(L.hkcsa_entropy_from_sa(_ptr(text), n, _ptr(sa), int(k), out, _ptr(scratch), nbytes, _stream()))
    return {"hk": (out[0] - out[1]) / n, "windows": int(out[2]), "contexts": int(out[3]), "grams": int(out[4])}


def lcp_arrays(text: torch.Tensor, sa: torch.Tensor, *, lcp: bool = True, plcp: bool = False,
               stats: list | None = None):
    """(LCP int32[n] in suffix-array order or None, PLCP int32[n] in text order or None) of `text` from its suffix
    array (csrc/lcp.cu).  stats: a list that receives [irreducible positions, sum of their values] (the call then
    waits for the device)."""
    if not (lcp or plcp):
        raise ValueError("ask for the LCP array, the PLCP array or both")
    L = _lib.load()
    n = text.numel()
    out_lcp = _empty(n, torch.int32, text.device) if lcp else None
    out_plcp = _empty(n, torch.int32, text.device) if plcp else None
    nbytes = L.hkcsa_lcp_scratch_bytes(n)
    scratch = _scratch(nbytes, text.device)
    h = (C.c_uint64 * 2)() if stats is not None else None
    check(L.hkcsa_lcp_build(_ptr(text), n, _ptr(sa), _ptr(out_lcp), _ptr(out_plcp), _ptr(scratch), nbytes, h,
                            _stream()))
    if stats is not None:
        stats[:] = [int(h[0]), int(h[1])]
    return out_lcp, out_plcp


def sort_pairs_u64(keys: torch.Tensor, vals: torch.Tensor, key_bits: int = 64):
    """In-place LSD onesweep radix sort of (int64-as-uint64 key, int32 value) pairs."""
    L = _lib.load()
    n = keys.numel()
    k2, v2 = torch.empty_like(keys), torch.empty_like(vals)
    nbytes = L.hkcsa_sort_scratch_bytes(n)
    scratch = _scratch(nbytes, keys.device)
    check(L.hkcsa_sort_pairs_u64(_ptr(keys), _ptr(vals), _ptr(k2), _ptr(v2), n, key_bits, _ptr(scratch), nbytes,
                                 _stream()))
    return keys, vals


def symbol_positions(bwt_sym: torch.Tensor):
    """FMIndex.precompute_rank (csa/csa.py:13-19): (positions int32[n] grouped by byte, start uint64[257] host)."""
    L = _lib.load()
    n = bwt_sym.numel()
    pos = _empty(n, torch.int32, bwt_sym.device)
    start = torch.zeros(257, dtype=torch.int64, device=bwt_sym.device)
    nbytes = L.hkcsa_symbol_positions_scratch_bytes(n)
    scratch = _scratch(nbytes, bwt_sym.device)
    check(L.hkcsa_symbol_positions(_ptr(bwt_sym), n, _ptr(pos), _ptr(start), _ptr(scratch), nbytes, _stream()))
    return pos, start.cpu().numpy().astype(np.uint64)


# ------------------------------------------------------------------ K3
class DeviceWaveletTree:
    """Level-wise wavelet tree with rank/select directories, resident in one device blob."""

    def __init__(self, sym: torch.Tensor, hist: np.ndarray | None = None):
        L = _lib.load()
        self.device = sym.device
        self.n = sym.numel()
        hist = byte_hist(sym) if hist is None else np.ascontiguousarray(hist, dtype=np.uint64)
        self.hist = hist
        self.plan = WtPlan()
        check(L.hkcsa_wt_plan_from_hist(hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(self.plan)))
        self.blob = torch.empty(int(self.plan.blob_bytes), dtype=torch.uint8, device=self.device)   # zeroed by the build
        scratch = _scratch(self.plan.scratch_bytes, self.device)
        check(L.hkcsa_wt_build(_ptr(sym), C.byref(self.plan), _ptr(self.blob), _ptr(scratch),
                               int(self.plan.scratch_bytes), _stream()))

    # -- shape
    @property
    def levels(self) -> int:
        return int(self.plan.levels)

    @property
    def sigma(self) -> int:
        return int(self.plan.sigma)

    @property
    def alphabet(self) -> bytes:
        return bytes(self.plan.sym_of_code[: self.sigma])

    def level_len(self, level: int) -> int:
        return int(self.plan.level_len[level])

    def level_ones(self, level: int) -> int:
        return int(self.plan.level_ones[level])

    def count_table(self) -> dict:
        """C[] as build_count returns it: {chr(byte): number of smaller symbols} (utils/utils.py:16-24)."""
        return {chr(self.plan.sym_of_code[c]): int(self.plan.C[c]) for c in range(self.sigma)}

    # -- bit-vector queries on one level
    def _u64(self, x) -> torch.Tensor:
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=torch.int64).contiguous()
        return torch.as_tensor(np.asarray(x, dtype=np.int64), device=self.device)

    def bv_rank(self, level: int, pos) -> torch.Tensor:
        pos = self._u64(pos)
        out = torch.empty_like(pos)
        check(_lib.load().hkcsa_bv_rank_batch(_ptr(self.blob), C.byref(self.plan), level, _ptr(pos), pos.numel(),
                                              _ptr(out), _stream()))
        return out

    def bv_select(self, level: int, k) -> torch.Tensor:
        k = self._u64(k)
        out = torch.empty_like(k)
        check(_lib.load().hkcsa_bv_select_batch(_ptr(self.blob), C.byref(self.plan), level, _ptr(k), k.numel(),
                                                _ptr(out), _stream()))
        return out

    def bv_bits(self, level: int, begin: int, count: int) -> torch.Tensor:
        out = _empty(count, torch.uint8, self.device)
        check(_lib.load().hkcsa_bv_unpack(_ptr(self.blob), C.byref(self.plan), level, begin, count, _ptr(out),
                                          _stream()))
        return out

    def bv_rank_range(self, level: int, begin: int, count: int) -> torch.Tensor:
        out = _empty(count, torch.int32, self.device)
        check(_lib.load().hkcsa_bv_rank_range(_ptr(self.blob), C.byref(self.plan), level, begin, count, _ptr(out),
                                              _stream()))
        return out

    # -- symbol-level queries
    def rank(self, sym, pos) -> torch.Tensor:
        """occ[c][i] (utils/utils.py:26-32): occurrences of byte sym[q] before position pos[q]."""
        pos = self._u64(pos)
        if isinstance(sym, torch.Tensor):
            sym = sym.to(device=self.device, dtype=torch.uint8).contiguous()
        else:
            sym = torch.as_tensor(np.asarray(sym, dtype=np.uint8), device=self.device)
        if sym.numel() != pos.numel():
            raise ValueError("sym and pos must have the same length")
        out = torch.empty_like(pos)
        check(_lib.load().hkcsa_wt_rank_batch(_ptr(self.blob), C.byref(self.plan), _ptr(sym), _ptr(pos), pos.numel(),
                                              _ptr(out), _stream()))
        return out

    def access(self, pos) -> torch.Tensor:
        pos = self._u64(pos)
        out = _empty(pos.numel(), torch.uint8, self.device)
        check(_lib.load().hkcsa_wt_access_batch(_ptr(self.blob), C.byref(self.plan), _ptr(pos), pos.numel(),
                                                _ptr(out), _stream()))
        return out

    def golomb(self, level: int, nbits: int, m: int) -> torch.Tensor:
        """GolombRiceEncoder.encode (csa/wavelet_tree.py:40-63) of bits [0, nbits) of a level -> uint8 0/1."""
        L = _lib.load()
        nbytes = L.hkcsa_golomb_scratch_bytes(nbits)
        scratch = _scratch(nbytes, self.device)
        total = C.c_uint64(0)
        check(L.hkcsa_golomb_encode(_ptr(self.blob), C.byref(self.plan), level, nbits, m, 0, 0, C.byref(total),
                                    _ptr(scratch), nbytes, _stream()))
        out = _empty(total.value, torch.uint8, self.device)
        if total.value:
            check(L.hkcsa_golomb_encode(_ptr(self.blob), C.byref(self.plan), level, nbits, m, _ptr(out), total.value,
                                        C.byref(total), _ptr(scratch), nbytes, _stream()))
        return out


# ------------------------------------------------------------------ entropy-coded bit-vectors (csrc/rrr.cu)
_RRR_TABLES: dict = {}


def rrr_tables(device) -> torch.Tensor:
    """The class / offset tables of the 15-bit block code, one copy per device."""
    key = torch.device(device).index
    if key not in _RRR_TABLES:
        L = _lib.load()
        t = torch.empty(L.hkcsa_rrr_tables_bytes(), dtype=torch.uint8, device=device)
        check(L.hkcsa_rrr_tables_init(_ptr(t), _stream()))
        _RRR_TABLES[key] = t
    return _RRR_TABLES[key]


class RrrVector:
    """A level of a wavelet tree (or a stand-alone DeviceBitVector) in the class/offset code: n*H_0 + o(n) bits,
    rank answered on the coded form, decodable bit for bit."""

    def __init__(self, plan: RrrPlan, blob: torch.Tensor):
        self.plan, self.blob = plan, blob

    @classmethod
    def encode(cls, wt: "DeviceWaveletTree", level: int, nbits: int | None = None) -> "RrrVector":
        L = _lib.load()
        nbits = wt.level_len(level) if nbits is None else int(nbits)
        tab = rrr_tables(wt.device)
        plan = RrrPlan()
        nscr = L.hkcsa_rrr_scratch_bytes(nbits)
        scratch = _scratch(nscr, wt.device)
        check(L.hkcsa_rrr_encode(_ptr(wt.blob), C.byref(wt.plan), level, nbits, _ptr(tab), C.byref(plan), None, 0,
                                 _ptr(scratch), nscr, _stream()))
        blob = torch.empty(max(int(plan.blob_bytes), 256), dtype=torch.uint8, device=wt.device)
        check(L.hkcsa_rrr_encode(_ptr(wt.blob), C.byref(wt.plan), level, nbits, _ptr(tab), C.byref(plan), _ptr(blob),
                                 blob.numel(), _ptr(scratch), nscr, _stream()))
        return cls(plan, blob[: max(int(plan.blob_bytes), 1)])

    @property
    def nbits(self) -> int:
        return int(self.plan.nbits)

    @property
    def coded_bits(self) -> int:
        """4 class bits per block + the offset stream + 64 bits per superblock of 960 bits."""
        return 4 * int(self.plan.nblocks) + int(self.plan.stream_bits) + 64 * int(self.plan.nsuper)

    def rank(self, pos) -> torch.Tensor:
        pos = (pos.to(device=self.blob.device, dtype=torch.int64).contiguous() if isinstance(pos, torch.Tensor)
               else torch.as_tensor(np.asarray(pos, dtype=np.int64), device=self.blob.device))
        out = torch.empty_like(pos)
        check(_lib.load().hkcsa_rrr_rank_batch(_ptr(self.blob), C.byref(self.plan), _ptr(rrr_tables(self.blob.device)),
                                               _ptr(pos), pos.numel(), _ptr(out), _stream()))
        return out

    def bits(self, begin: int = 0, count: int | None = None) -> torch.Tensor:
        count = self.nbits - begin if count is None else count
        out = _empty(count, torch.uint8, self.blob.device)
        check(_lib.load().hkcsa_rrr_unpack(_ptr(self.blob), C.byref(self.plan), _ptr(rrr_tables(self.blob.device)),
                                           begin, count, _ptr(out), _stream()))
        return out


def wt_from_coded_levels(plan: WtPlan, coded: list, device) -> DeviceWaveletTree:
    """Rebuild the query blob of a wavelet tree from its RRR-coded levels: node tables from the plan, payload bits
    decoded in place, block headers / superblocks / select samples recomputed (checked against the plan's counts)."""
    L = _lib.load()
    wt = DeviceWaveletTree.__new__(DeviceWaveletTree)
    wt.device, wt.n, wt.hist, wt.plan = torch.device(device), int(plan.n), None, plan
    wt.blob = torch.empty(int(plan.blob_bytes), dtype=torch.uint8, device=device)
    check(L.hkcsa_wt_restore_begin(C.byref(plan), _ptr(wt.blob), _stream()))
    tab = rrr_tables(device)
    for level, vec in enumerate(coded):
        if isinstance(vec, np.ndarray):             # a level kept plain: payload words back behind zeroed headers
            a, b = int(plan.off_blocks[level]), int(plan.off_super[level])
            rows = torch.zeros(((b - a) // 32, 8), dtype=torch.int32, device=device)
            k = min(rows.shape[0], vec.shape[0])
            rows[:k, 1:] = torch.from_numpy(vec[:k].view(np.int32)).to(device)
            wt.blob[a:a + rows.numel() * 4] = rows.view(torch.uint8).reshape(-1)
            continue
        check(L.hkcsa_rrr_restore_level(_ptr(vec.blob), C.byref(vec.plan), _ptr(tab), C.byref(plan), level,
                                        _ptr(wt.blob), _stream()))
    scratch = _scratch(plan.scratch_bytes, device)
    check(L.hkcsa_wt_restore_finish(C.byref(plan), _ptr(wt.blob), _ptr(scratch), int(plan.scratch_bytes), _stream()))
    return wt


class DeviceBitVector(DeviceWaveletTree):
    """Stand-alone rank/select bit-vector (SuccinctRankSelect, csa/wavelet_tree.py:5-25): a one-level
    plan whose level 0 is the bitmap.  `bits`: uint8 device tensor, one byte per bit."""

    def __init__(self, bits: torch.Tensor):  # noqa: super().__init__ builds a tree; this builds one level
        L = _lib.load()
        self.device = bits.device
        self.n = bits.numel()
        self.hist = None
        self.plan = WtPlan()
        check(L.hkcsa_bitvec_plan(self.n, C.byref(self.plan)))
        self.blob = torch.zeros(int(self.plan.blob_bytes), dtype=torch.uint8, device=self.device)
        scratch = _scratch(self.plan.scratch_bytes, self.device)
        check(L.hkcsa_bitvec_build(_ptr(bits), C.byref(self.plan), _ptr(self.blob), _ptr(scratch),
                                   int(self.plan.scratch_bytes), _stream()))

    @property
    def ones(self) -> int:
        return int(self.plan.level_ones[0])


def partition_bytes(seq: torch.Tensor, lut: np.ndarray):
    """Stable bucket partition of a byte sequence by lut[byte] -> (partitioned uint8[n], sizes uint64[256])."""
    L = _lib.load()
    n = seq.numel()
    lut = np.ascontiguousarray(lut, dtype=np.uint8)
    out = _empty(n, torch.uint8, seq.device)
    sizes = np.zeros(256, dtype=np.uint64)
    nbytes = L.hkcsa_partition_scratch_bytes(n)
    scratch = _scratch(nbytes, seq.device)
    check(L.hkcsa_partition_bytes(_ptr(seq), n, lut.ctypes.data_as(C.POINTER(C.c_uint8)), _ptr(out),
                                  sizes.ctypes.data_as(C.POINTER(C.c_uint64)), _ptr(scratch), nbytes, _stream()))
    return out, sizes


# ------------------------------------------------------------------ K4
@dataclass
class SampledSA:
    plan: SsaPlan
    blob: torch.Tensor


def build_sampled_sa(sa: torch.Tensor, rate: int) -> SampledSA:
    L = _lib.load()
    plan = SsaPlan()
    check(L.hkcsa_ssa_plan_make(sa.numel(), rate, C.byref(plan)))
    blob = torch.zeros(int(plan.blob_bytes), dtype=torch.uint8, device=sa.device)
    scratch = _scratch(plan.scratch_bytes, sa.device)
    check(L.hkcsa_ssa_build(_ptr(sa), C.byref(plan), _ptr(blob), _ptr(scratch), int(plan.scratch_bytes), _stream()))
    return SampledSA(plan, blob)


def pack_patterns_host(patterns):
    """list[str|bytes] -> (bytes of all patterns back to back, int64[P+1] offsets), on the host.  A list of latin-1
    str patterns (what the reference's find_range takes, csa/enhanced_fm_index.py:21) is packed by ONE join + ONE
    encode and a C-level len() map; anything else goes pattern by pattern (a str beyond latin-1 raises
    UnicodeEncodeError there: the caller decides what such a pattern means)."""
    P = len(patterns)
    flat = None
    try:
        joined = "".join(patterns)                      # TypeError unless every pattern is a str
        flat = joined.encode("latin-1")                 # UnicodeEncodeError beyond latin-1: the slow path reports it
        lens = np.fromiter(map(len, patterns), dtype=np.int64, count=P)
    except (TypeError, UnicodeEncodeError):
        flat = None
    if flat is None:
        enc = [p.encode("latin-1") if isinstance(p, str) else bytes(p) for p in patterns]
        lens = np.fromiter(map(len, enc), dtype=np.int64, count=P)
        flat = b"".join(enc)
    off = np.zeros(P + 1, dtype=np.int64)
    if P:
        np.cumsum(lens, out=off[1:])
    return flat, off


def pack_patterns(patterns, device=None):
    """list[str|bytes] -> (uint8[sum m], int64[P+1]) on the device (pack_patterns_host + two staged copies)."""
    device = device or _require_cuda()
    flat, off = pack_patterns_host(patterns)
    return to_device_u8(flat, device), to_device_u8(off.view(np.uint8), device).view(torch.int64)


# ------------------------------------------------------------------ query plumbing of DeviceIndex and MultiSliceIndex
def _expand_ranges(lo: torch.Tensor, hi: torch.Tensor, wide: bool):
    """SA ranges (lo, hi; -1: no match) -> (CSR offsets int64[P+1], their rows in SA order: int32, int64 if wide)."""
    L = _lib.load()
    P = lo.numel()
    cnt = torch.where(lo >= 0, hi - lo + 1, torch.zeros_like(lo))       # plumbing: CSR offsets
    out_off = torch.zeros(P + 1, dtype=torch.int64, device=lo.device)
    out_off[1:] = torch.cumsum(cnt, 0)
    total = int(out_off[-1].item()) if P else 0
    rows = _empty(total, torch.int64 if wide else torch.int32, lo.device)
    expand = L.hkcsa_expand_ranges64 if wide else L.hkcsa_expand_ranges
    check(expand(_ptr(lo), _ptr(hi), _ptr(out_off), P, _ptr(rows), _stream()))
    return out_off, rows


def _extract_requests(begin, end, n: int, device):
    """The requests of an extract batch -> (begin, end as int64 device tensors, out_off int64[R+1], out uint8[total]),
    once 0 <= begin <= end <= n is checked (one read-back).  An empty `out` is already the answer."""
    begin = begin.to(device=device, dtype=torch.int64).contiguous()
    end = end.to(device=device, dtype=torch.int64).contiguous()
    if begin.shape != end.shape or begin.dim() != 1:
        raise ValueError("begin and end must be 1-d tensors of the same length")
    R = begin.numel()
    out_off = torch.zeros(R + 1, dtype=torch.int64, device=device)
    if R == 0:
        return begin, end, out_off, _empty(0, torch.uint8, device)
    out_off[1:] = torch.cumsum(end - begin, 0)                          # plumbing: CSR offsets
    bad = ((begin < 0) | (end < begin) | (end > n)).any()
    total, bad = torch.stack([out_off[-1], bad.to(torch.int64)]).tolist()   # one read-back for both
    if bad:
        raise ValueError(f"extract ranges must satisfy 0 <= begin <= end <= n = {n}")
    return begin, end, out_off, _empty(total, torch.uint8, device)


@dataclass
class BuildStats:
    sa: SaStats = field(default_factory=SaStats)
    n: int = 0


class DeviceIndex:
    """FM index over `text` exactly as given (callers append the sentinel: EnhancedFMIndex adds '$',
    csa/enhanced_fm_index.py:9).  Everything stays on the device."""

    def __init__(self, text: torch.Tensor, *, sa_sample_rate: int = 0, keep_sa: bool = True,
                 keep_text: bool = True, host_sa: torch.Tensor | None = None,
                 host_bwt: torch.Tensor | None = None):
        """host_sa / host_bwt: optional pinned host tensors (int32[n] / uint8[n]) that receive the suffix
        array and the BWT; the copies run on a side stream and overlap the rest of the build.  The
        caller synchronises (torch.cuda.synchronize()) before reading them."""
        _require_cuda()
        L = _lib.load()
        dev = self.device = text.device
        n = self.n = text.numel()
        self.stats = BuildStats(n=n)
        if n > _lib.MAX_N:
            raise HkcsaError(_lib.ERANGE, f"text of {n} symbols exceeds the single-GPU limit {_lib.MAX_N}")
        # Every buffer is in place before the first kernel: the whole build is ONE library call (hkcsa_index_build:
        # suffix array + BWT, then the wavelet tree on a high-priority stream beside the sampled suffix array), so no
        # Python runs while the GPU could be working.  The tree's shape depends on the byte histogram, which the call
        # computes itself: the blob is allocated at the bound for n symbols and trimmed to the plan's size afterwards.
        main = torch.cuda.current_stream()
        self.sa = _empty(n, torch.int32, dev)
        self.bwt = _empty(n, torch.uint8, dev)
        sa_bytes = L.hkcsa_sa_scratch_bytes(n)
        sa_scratch = _scratch(sa_bytes, dev)
        blob_cap, wt_cap = int(L.hkcsa_wt_blob_bound(n)), int(L.hkcsa_wt_scratch_bound(n))
        blob = torch.empty(blob_cap, dtype=torch.uint8, device=dev)       # zeroed by the build
        wt_scratch = _scratch(wt_cap, dev)
        wt = DeviceWaveletTree.__new__(DeviceWaveletTree)
        wt.device, wt.n, wt.plan = dev, n, WtPlan()
        self.ssa = None
        ssa_plan = ssa_blob = ssa_scratch = None
        crit = ssa_stream = main
        if sa_sample_rate > 0:
            ssa_plan = SsaPlan()
            check(L.hkcsa_ssa_plan_make(n, sa_sample_rate, C.byref(ssa_plan)))
            ssa_blob = torch.zeros(int(ssa_plan.blob_bytes), dtype=torch.uint8, device=dev)
            ssa_scratch = _scratch(ssa_plan.scratch_bytes, dev)
            # the tree is the critical path of the tail: on a high-priority stream the block scheduler serves it first
            # and the sampled-SA kernel fills what is left (tree alone 2.6 ms at C3; sharing the SMs evenly 3.4 ms)
            crit = _aux_stream(dev, "critical", priority=-1)
            ssa_stream = _aux_stream(dev, "ssa")
            tail = os.environ.get("HKCSA_TAIL", "")              # experiment knob: how the tail shares the GPU
            if tail == "flat":
                crit = main
            elif tail == "serial":
                crit = ssa_stream = main
            elif tail == "ssa_high":
                crit, ssa_stream = _aux_stream(dev, "ssa"), _aux_stream(dev, "critical", priority=-1)
        check(L.hkcsa_index_build(_ptr(text), n, _ptr(self.sa), _ptr(self.bwt), _ptr(sa_scratch), sa_bytes,
                                  C.byref(wt.plan), _ptr(blob), blob_cap, _ptr(wt_scratch), wt_cap,
                                  C.byref(ssa_plan) if ssa_plan is not None else None, _ptr(ssa_blob), _ptr(ssa_scratch),
                                  int(ssa_plan.scratch_bytes) if ssa_plan is not None else 0,
                                  main.cuda_stream, crit.cuda_stream if crit is not main else None,
                                  ssa_stream.cuda_stream if ssa_stream is not main else None, C.byref(self.stats.sa)))
        if crit is not main:
            for t in (self.bwt, blob, wt_scratch):
                t.record_stream(crit)
            for t in (self.sa, ssa_blob, ssa_scratch):
                t.record_stream(ssa_stream)
        used = int(wt.plan.blob_bytes)
        # keep exactly the plan's bytes: a view while most of the bound is in use, a copy (and the bound released) otherwise
        wt.blob = blob[:used] if 4 * used >= 3 * blob_cap else blob[:used].clone()
        wt.hist = np.ctypeslib.as_array(self.stats.sa.byte_hist).copy()
        self.wt = wt
        if ssa_plan is not None:
            self.ssa = SampledSA(ssa_plan, ssa_blob)
        side = None
        if host_sa is not None or host_bwt is not None:
            side = _aux_stream(dev, "copy")
            side.wait_stream(main)
            with torch.cuda.stream(side):
                if host_sa is not None:
                    host_sa.copy_(self.sa, non_blocking=True)
                if host_bwt is not None:
                    host_bwt.copy_(self.bwt, non_blocking=True)
            self.sa.record_stream(side)        # keep_sa=False must not hand the buffer back while the copy runs
            self.bwt.record_stream(side)
        self._side = side
        self.text = text if keep_text else None
        if not keep_sa:
            if self.ssa is None:
                raise ValueError("dropping the suffix array needs sa_sample_rate > 0")
            self.sa = None

    @classmethod
    def from_parts(cls, n: int, plan: WtPlan, blob: torch.Tensor, ssa: "SampledSA | None"):
        """A query-only replica assembled from a broadcast wavelet-tree blob (hkcsa.dist)."""
        self = cls.__new__(cls)
        self.device = blob.device
        self.n = n
        self.stats = BuildStats(n=n)
        self.sa = None
        self.bwt = None
        self.text = None
        self.wt = DeviceWaveletTree.__new__(DeviceWaveletTree)
        self.wt.device, self.wt.n, self.wt.hist, self.wt.plan, self.wt.blob = blob.device, n, None, plan, blob
        self.ssa = ssa
        return self

    # -- persistence (the reference never writes its index to disk: SURVEY.md section 5; next-row 3)
    def coded_levels(self) -> list:
        """Every wavelet-tree level in the class/offset code (csrc/rrr.cu), cached."""
        if getattr(self, "_coded", None) is None:
            self._coded = [RrrVector.encode(self.wt, l) for l in range(self.wt.levels)]
        return self._coded

    def space(self) -> dict:
        """Bits per symbol of the index: the query blob as it lives in HBM, and the entropy-coded form save() writes."""
        n = max(self.n, 1)
        coded = self.coded_levels()
        ssa_bits = 8 * int(self.ssa.blob.numel()) if self.ssa is not None else 0
        raw = [self.wt.level_len(l) for l in range(self.wt.levels)]
        stored = [min(v.coded_bits, r) for v, r in zip(coded, raw)]       # a level the code does not shrink stays plain
        return {"n": self.n, "levels": self.wt.levels,
                "query_blob_bits_per_symbol": 8.0 * self.wt.blob.numel() / n,
                "raw_level_bits_per_symbol": sum(raw) / n,
                "coded_level_bits_per_symbol": sum(stored) / n,
                "coded_bits_per_level": [v.coded_bits for v in coded],
                "stored_bits_per_level": stored,
                "levels_kept_plain": [l for l, (v, r) in enumerate(zip(coded, raw)) if v.coded_bits >= r],
                "sampled_sa_bits_per_symbol": ssa_bits / n}

    def save(self, path: str, compressed: bool = False, extra: dict | None = None) -> None:
        """Write the query structures to one .npz file.  compressed=False: the wavelet-tree blob exactly as it lives
        in HBM (loading is a single host->device copy).  compressed=True: every level in the class/offset code
        (n*H_0 of the level + o(n) bits; over the levels of a BWT: n*H_k + o(n)); load() decodes the payload bits
        in place and rebuilds the rank directories -- the restored blob is bit-identical.  extra: more named arrays
        for the same file (a caller's metadata); load() reads its own keys by name and ignores them."""
        parts = {"n": np.array([self.n], dtype=np.int64),
                 "wt_plan": np.frombuffer(bytes(self.wt.plan), dtype=np.uint8)}
        if compressed:
            for l, vec in enumerate(self.coded_levels()):
                if vec.coded_bits < self.wt.level_len(l):
                    parts[f"rrr_plan_{l}"] = np.frombuffer(bytes(vec.plan), dtype=np.uint8)
                    parts[f"rrr_blob_{l}"] = to_host(vec.blob)
                else:       # the code does not shrink this level: its 224 payload bits per rank block, headers dropped
                    a, b = int(self.wt.plan.off_blocks[l]), int(self.wt.plan.off_super[l])
                    words = self.wt.blob[a:b].cpu().numpy().view(np.uint32).reshape(-1, 8)
                    parts[f"raw_payload_{l}"] = np.ascontiguousarray(words[:, 1:])
        else:
            parts["wt_blob"] = to_host(self.wt.blob)
        if self.ssa is not None:
            parts["ssa_plan"] = np.frombuffer(bytes(self.ssa.plan), dtype=np.uint8)
            parts["ssa_blob"] = to_host(self.ssa.blob)
        for key, arr in (extra or {}).items():
            if key in parts:
                raise ValueError(f"extra key {key!r} collides with an index array")
            parts[key] = np.asarray(arr)
        with open(path, "wb") as f:
            np.savez(f, **parts)

    @classmethod
    def load(cls, path: str, device=None) -> "DeviceIndex":
        device = device or _require_cuda()
        z = np.load(path)
        plan = WtPlan.from_buffer_copy(z["wt_plan"].tobytes())
        if "wt_blob" in z.files:
            blob = to_device_u8(z["wt_blob"], device)
        else:
            coded = []
            for l in range(int(plan.levels)):
                if f"rrr_plan_{l}" in z.files:
                    rp = RrrPlan.from_buffer_copy(z[f"rrr_plan_{l}"].tobytes())
                    coded.append(RrrVector(rp, torch.from_numpy(z[f"rrr_blob_{l}"]).to(device)))
                else:
                    coded.append(np.asarray(z[f"raw_payload_{l}"], dtype=np.uint32))
            blob = wt_from_coded_levels(plan, coded, device).blob
        ssa = None
        if "ssa_plan" in z.files:
            ssa = SampledSA(SsaPlan.from_buffer_copy(z["ssa_plan"].tobytes()), torch.from_numpy(z["ssa_blob"]).to(device))
        return cls.from_parts(int(z["n"][0]), plan, blob, ssa)

    # k-mer jump table (query accelerator, built on first use for large batches)
    KMER_MIN_BATCH = 1 << 18
    OCC_MIN_BATCH = 1 << 20      # batches from which count_batch builds the sampled Occ table on its own

    def build_kmer_table(self):
        """SA ranges of every k-mer over the alphabet (k = largest with sigma^k <= 2^21), computed by the count
        kernel itself; count_batch then starts each pattern from the entry of its last k symbols."""
        L = _lib.load()
        k = int(L.hkcsa_kmer_k(self.wt.sigma))
        if k == 0:
            self._kmer = (None, 0)
            return self._kmer
        entries = int(L.hkcsa_kmer_entries(self.wt.sigma, k))
        table = torch.empty(entries * 2, dtype=torch.int32, device=self.device)
        nbytes = L.hkcsa_kmer_scratch_bytes(self.wt.sigma, k)
        scratch = _scratch(nbytes, self.device)
        check(L.hkcsa_kmer_table_build(_ptr(self.wt.blob), C.byref(self.wt.plan), k, _ptr(table), _ptr(scratch), nbytes,
                                       _stream()))
        self._kmer = (table, k)
        return self._kmer

    def entropy(self, k: int) -> float:
        """H_k (bits per symbol) of the indexed text, from the suffix array of the build."""
        if self.sa is None or self.text is None:
            raise ValueError("H_k is computed from the text and the suffix array, which this index no longer holds")
        return entropy_from_sa(self.text, self.sa, k)["hk"]

    # LCP (csrc/lcp.cu): from the text and the suffix array, or from Sadakane's 2n-bit encoding once those are gone
    def _lcp_source(self):
        if self.sa is None or self.text is None:
            raise ValueError("the LCP array is computed from the text and the suffix array, which this index no "
                             "longer holds")
        return self.text, self.sa

    def lcp(self) -> torch.Tensor:
        """int32[n]: LCP[0] = 0, LCP[r] = longest common prefix of the suffixes in rows r-1 and r.  Not cached."""
        return lcp_arrays(*self._lcp_source(), lcp=True)[0]

    def plcp(self) -> torch.Tensor:
        """int32[n]: PLCP[i] = LCP[ISA[i]], the LCP array in text order.  Not cached."""
        return lcp_arrays(*self._lcp_source(), lcp=False, plcp=True)[1]

    def build_lcp_bits(self) -> None:
        """Sadakane's encoding of PLCP for lcp_rows, built while the text and the suffix array are at hand: a bit
        vector H with a one at PLCP[i] + 2i for every i (n ones in < 2n bits).  H is kept as at most two
        DeviceBitVectors split at HKCSA_MAX_N bits (the limit of one bit vector)."""
        plcp = self.plcp()
        bits = _empty(2 * self.n, torch.uint8, self.device)
        check(_lib.load().hkcsa_plcp_bits(_ptr(plcp), self.n, _ptr(bits), _stream()))
        del plcp
        cut = _lib.MAX_N
        self._lcp_bits = [DeviceBitVector(bits[a:a + cut]) for a in range(0, max(bits.numel(), 1), cut)]

    def _lcp_bits_held(self) -> int:
        """Bits held by the LCP encoding (rank blocks and directories of H); 0 before build_lcp_bits()."""
        return sum(8 * int(v.blob.numel()) for v in getattr(self, "_lcp_bits", None) or [])

    def _plcp_decode(self, pos: torch.Tensor) -> torch.Tensor:
        """int64 PLCP[pos] from H: select(H, i + 1) - 1 - 2i, the select on the piece that holds the (i+1)-th one."""
        pieces = self._lcp_bits
        k = pos + 1
        sel = pieces[0].bv_select(0, k)
        if len(pieces) == 2:
            first = pieces[0].ones
            sel2 = pieces[1].bv_select(0, (k - first).clamp(min=1)) + _lib.MAX_N
            sel = torch.where(k > first, sel2, sel)
        return sel - 1 - 2 * pos

    def lcp_rows(self, rows: torch.Tensor, *, use_samples: bool | None = None) -> torch.Tensor:
        """int32: LCP[rows] from the encoding of build_lcp_bits(): LCP[r] = PLCP[locate(r)], the locate of
        locate_rows (sampled or full suffix array, as it chooses)."""
        if getattr(self, "_lcp_bits", None) is None:
            raise ValueError("no LCP encoding: call build_lcp_bits() while the index holds its text and suffix array")
        rows = rows.to(device=self.device, dtype=torch.int32).contiguous()
        pos = self.locate_rows(rows, use_samples=use_samples).to(torch.int64)
        return self._plcp_decode(pos).to(torch.int32)

    def psi(self) -> torch.Tensor:
        """The Psi function of the compressed suffix array (Grossi-Vitter; README.md:4 of the reference): psi[i] =
        the row of the suffix that starts one symbol later, SA[psi[i]] = SA[i] + 1 (mod n), i.e. the inverse of LF.
        It is the concatenation, over the symbols in order, of FMIndex.precompute_rank's ascending position lists
        (csa/csa.py:13-19) -- one stable partition of the row numbers by BWT symbol (hkcsa_symbol_positions)."""
        if self.bwt is None:
            raise ValueError("psi is derived from the BWT, which this index no longer holds")
        return symbol_positions(self.bwt)[0]

    def build_occ_table(self, shift: int = 5, bwt: torch.Tensor | None = None, layout: int = 0):
        """Sampled Occ table (csrc/occ_table.cu): the reference's dense occ (utils/utils.py:26-32) kept at every
        2^shift-th row next to the BWT bytes of that stretch.  Optional: costs 2^shift + 4 sigma bytes per 2^shift
        rows, makes a rank one or two sector reads instead of one per wavelet level.  layout=1: per-symbol
        bitmaps, one 8-byte entry per symbol and 32 rows (8 sigma bytes per 32 rows): a rank is a single memory
        request.  Needs the BWT (kept by the builder; replicas pass it in)."""
        L = _lib.load()
        bwt = self.bwt if bwt is None else bwt
        if bwt is None:
            raise ValueError("the sampled Occ table is built from the BWT, which this index no longer holds")
        plan = OccPlan()
        check(L.hkcsa_occ_plan_make(self.n, self.wt.sigma, shift, layout, C.byref(plan)))
        blob = _empty(int(plan.blob_bytes), torch.uint8, self.device)
        scratch = _scratch(int(plan.scratch_bytes), self.device)
        check(L.hkcsa_occ_build(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(bwt), C.byref(plan), _ptr(blob),
                                _ptr(scratch), int(plan.scratch_bytes), _stream()))
        self._occ = (plan, blob)
        return self._occ

    # find_range, batched (csa/enhanced_fm_index.py:21-32)
    def count_batch(self, pat: torch.Tensor, off: torch.Tensor, use_kmer_table: bool | None = None,
                    use_occ_table: bool | None = None):
        """use_occ_table: None = use the sampled Occ table when one was built (build_occ_table) or build it for a
        batch of OCC_MIN_BATCH patterns or more; False = always rank on the wavelet tree.  Identical ranges."""
        P = off.numel() - 1
        lo = _empty(P, torch.int64, self.device)
        hi = _empty(P, torch.int64, self.device)
        if self.n == 0:
            raise ValueError("empty index")
        if use_kmer_table is None:
            use_kmer_table = getattr(self, "_kmer", None) is not None or P >= self.KMER_MIN_BATCH
        table, k = (None, 0)
        if use_kmer_table:
            table, k = getattr(self, "_kmer", None) or self.build_kmer_table()
        occ = getattr(self, "_occ", None)
        if use_occ_table is None:
            # large batches amortise the table (0.5-2 ms to build) many times over: build it when the BWT is at
            # hand and the table takes at most a quarter of the free device memory
            if occ is None and P >= self.OCC_MIN_BATCH and self.bwt is not None:
                need = 8 * self.wt.sigma * (self.n // 32 + 4) + self.n
                if need <= torch.cuda.mem_get_info(self.device)[0] // 4:
                    occ = self.build_occ_table(5, layout=1)
            use_occ_table = occ is not None
        if use_occ_table:
            if occ is None:
                raise ValueError("no sampled Occ table: call build_occ_table() first")
            check(_lib.load().hkcsa_count_batch_occ(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(occ[1]),
                                                    C.byref(occ[0]), _ptr(table), k, _ptr(pat), _ptr(off), P,
                                                    _ptr(lo), _ptr(hi), _stream()))
            return lo, hi
        check(_lib.load().hkcsa_count_batch_kmer(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(table), k, _ptr(pat),
                                                 _ptr(off), P, _ptr(lo), _ptr(hi), _stream()))
        return lo, hi

    def count_batch_peers(self, pat: torch.Tensor, off: torch.Tensor, out_base: int, peer_lo, peer_hi,
                          use_kmer_table: bool | None = None) -> None:
        """count_batch for one rank's slice of a global batch, the gather fused into the search: the ranges are
        written at [out_base + p] of the lo / hi arrays of every rank (peer_lo / peer_hi: ctypes uint64 arrays of
        peer-mapped device pointers, hkcsa.dist.PeerRanges).  Ranks on the sampled Occ table when one was built."""
        P = off.numel() - 1
        if self.n == 0:
            raise ValueError("empty index")
        if use_kmer_table is None:
            use_kmer_table = getattr(self, "_kmer", None) is not None or P >= self.KMER_MIN_BATCH
        table, k = (None, 0)
        if use_kmer_table:
            table, k = getattr(self, "_kmer", None) or self.build_kmer_table()
        occ = getattr(self, "_occ", None)
        check(_lib.load().hkcsa_count_batch_peers(
            _ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(occ[1]) if occ else None, C.byref(occ[0]) if occ else None,
            _ptr(table), k, _ptr(pat), _ptr(off), P, int(out_base), len(peer_lo), peer_lo, peer_hi, _stream()))

    # find, batched (csa/enhanced_fm_index.py:15-19): CSR (offsets, positions in SA order)
    def locate_batch(self, pat: torch.Tensor, off: torch.Tensor, *, use_samples: bool | None = None):
        out_off, rows = _expand_ranges(*self.count_batch(pat, off), wide=False)
        return out_off, self.locate_rows(rows, use_samples=use_samples)

    def locate_rows(self, rows: torch.Tensor, *, use_samples: bool | None = None) -> torch.Tensor:
        L = _lib.load()
        if use_samples is None:
            use_samples = self.sa is None
        out = _empty(rows.numel(), torch.int32, self.device)
        if use_samples:
            if self.ssa is None:
                raise ValueError("index was built without a sampled suffix array")
            if rows.numel() == 0:
                return out
            row0 = self.row_of_suffix0()
            occ = getattr(self, "_occ", None)
            if occ is not None:      # LF steps from the sampled Occ table: two sectors instead of one per level
                check(L.hkcsa_locate_rows_occ(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(occ[1]), C.byref(occ[0]),
                                              _ptr(self.ssa.blob), C.byref(self.ssa.plan), row0, _ptr(rows),
                                              rows.numel(), _ptr(out), _stream()))
                return out
            check(L.hkcsa_locate_rows(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(self.ssa.blob),
                                      C.byref(self.ssa.plan), row0, _ptr(rows), rows.numel(), _ptr(out), _stream()))
        else:
            check(L.hkcsa_gather_u32(_ptr(self.sa), _ptr(rows), rows.numel(), _ptr(out), _stream()))
        return out

    # extract (csrc/extract.cu): text[begin:end) from the index alone -- the reference's decompress returns ''
    def isa_samples(self) -> torch.Tensor:
        """int32[S + 1]: the row of the suffix at text position k * rate for k < S = ceil(n / rate), and [S] = [0].
        Derived from the sampled suffix array (no text, no full SA: a loaded index has it too); built on first use."""
        if getattr(self, "_isa", None) is None:
            if self.ssa is None:
                raise ValueError("index was built without a sampled suffix array")
            out = _empty(int(self.ssa.plan.n_samples) + 1, torch.int32, self.device)
            check(_lib.load().hkcsa_isa_samples(_ptr(self.ssa.blob), C.byref(self.ssa.plan), _ptr(out), _stream()))
            self._isa = out
        return self._isa

    def row_of_suffix0(self) -> int:
        """The row of suffix 0 (isa_samples()[0]): the LF step of a sampled locate needs it to be exact on a text that
        holds its last symbol elsewhere too.  Read back once per sampled suffix array."""
        if getattr(self, "_row0", None) is None or self._row0[0] is not self.ssa:
            self._row0 = (self.ssa, int(self.isa_samples()[0].item()))
        return self._row0[1]

    @property
    def invertible(self) -> bool:
        """Whether LF is the inverse of the suffix order on this index, i.e. whether extract gives back the text.  With
        j0 = the row of suffix 0 and c = bwt[j0] (= text[n-1]), LF is right everywhere iff j0 is the first row whose BWT
        symbol is c.  Always true with a unique sentinel; a text that holds the sentinel elsewhere may fail it."""
        if getattr(self, "_invertible", None) is None:
            if self.n == 0:
                self._invertible = False
            else:
                j0 = self.isa_samples()[:1].to(torch.int64)
                c = self.wt.access(j0)
                self._invertible = int(self.wt.rank(c, j0).item()) == 0
        return self._invertible

    def extract_batch(self, begin: torch.Tensor, end: torch.Tensor, *, use_occ_table: bool | None = None):
        """text[begin[q]:end[q]) for every q (int64 device tensors; 0 <= begin <= end <= n, sentinel included) ->
        (out_off int64[R+1], bytes uint8[total]) on the device, request q at bytes[out_off[q]:out_off[q+1]].
        use_occ_table: None = LF steps on the sampled Occ table when one was built (as locate_rows), else the tree."""
        L = _lib.load()
        if not self.invertible:
            raise ValueError("LF does not invert the suffix order on this index (its text holds the sentinel "
                             "elsewhere too): extract cannot give the text back")
        begin, end, out_off, out = _extract_requests(begin, end, self.n, self.device)
        if out.numel() == 0:
            return out_off, out
        R = begin.numel()
        occ = getattr(self, "_occ", None)
        if use_occ_table is None:
            use_occ_table = occ is not None
        if use_occ_table and occ is None:
            raise ValueError("no sampled Occ table: call build_occ_table() first")
        plan, blob = occ if use_occ_table else (None, None)
        isa = self.isa_samples()
        nbytes = L.hkcsa_extract_scratch_bytes(R)
        scratch = _scratch(nbytes, self.device)
        check(L.hkcsa_extract(_ptr(self.wt.blob), C.byref(self.wt.plan), _ptr(blob),
                              C.byref(plan) if plan is not None else None, _ptr(isa), int(self.ssa.plan.rate),
                              _ptr(begin), _ptr(end), _ptr(out_off), R, _ptr(out), _ptr(scratch), nbytes, _stream()))
        return out_off, out

    def extract(self, begin: int, end: int, *, use_occ_table: bool | None = None) -> torch.Tensor:
        """text[begin:end) of the indexed text (sentinel included) as a uint8 device tensor."""
        b = torch.tensor([begin], dtype=torch.int64, device=self.device)
        e = torch.tensor([end], dtype=torch.int64, device=self.device)
        return self.extract_batch(b, e, use_occ_table=use_occ_table)[1]


# ------------------------------------------------------------------ measurement hook
def prof_enable(on: bool, classes=None) -> None:
    """classes: names of the kernel classes to time (None = all)."""
    L = _lib.load()
    check(L.hkcsa_prof_reset())
    if on and classes:
        mask = 0
        for name in classes:
            idx = L.hkcsa_prof_class_index(name.encode())
            if idx < 0:
                raise ValueError(f"unknown kernel class {name!r}")
            mask |= 1 << idx
        check(L.hkcsa_prof_enable_classes(mask))
    else:
        check(L.hkcsa_prof_enable(1 if on else 0))


def prof_read() -> dict:
    L = _lib.load()
    arr = (_lib.ProfEntry * _lib.PROF_CLASSES)()
    n = C.c_int(0)
    check(L.hkcsa_prof_read(arr, _lib.PROF_CLASSES, C.byref(n)))
    out = {}
    for i in range(n.value):
        e = arr[i]
        if e.launches:
            out[e.name.decode()] = {"launches": int(e.launches), "ms": float(e.ms), "alg_bytes": int(e.alg_bytes)}
    check(L.hkcsa_prof_reset())
    return out
