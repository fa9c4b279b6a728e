"""Drop-in for the reference's csa/enhanced_fm_index.py on B200: ``EnhancedFMIndex`` (:7-40).

Same constructor, attributes (``text`` with the '$' sentinel, ``suffix_array``, ``bwt``,
``occ``, ``count``) and methods (``find``, ``find_range``, ``rank``).  The build runs
libhkcsa K1 -> K2 -> K3 on the device; ``occ`` is answered by rank queries on the wavelet
tree instead of the reference's dense n*sigma table (utils/utils.py:26-32); queries run
K4.  Batched entry points (``find_range_batch`` / ``count_batch`` / ``find_batch``) are
additions for the C4 workload: one kernel launch for any number of patterns.
"""
import numpy as np

from hkcsa import views as _views


class EnhancedFMIndex:
    def __init__(self, text):
        from hkcsa import engine
        self._E = engine
        self._smap = None
        if isinstance(text, str):
            self._text0, self._text = text, None                     # self.text = text + "$" (:9), built on first access
            self._smap = engine.SymbolMap(text, extra="$")           # identity for latin-1 text
            d_text = engine.to_device_u8(self._smap.host_bytes(text), tail=self._smap.encode("$"))
        else:                                                        # bytes / uint8 array / tensor (extension)
            import torch
            d_text = engine.to_device_u8(text, tail=b"$")
            self._text0, self._text = None, (d_text if isinstance(text, torch.Tensor) else bytes(text) + b"$")
        self._idx = engine.DeviceIndex(d_text)                       # :10-12 (SA, BWT, wavelet tree = occ)
        self._sa = None
        self._lcp = None
        self._bwt = None
        self._occ = None
        self._str = isinstance(text, str)
        self.count = self._idx.wt.count_table()                      # :13  build_count(self.text)
        if not self._str:
            self.count = {ord(k): v for k, v in self.count.items()}
        elif not self._smap.identity:
            self.count = {self._smap.symbol(ord(k)): v for k, v in self.count.items()}

    # ---- attributes of the reference, materialised on first use
    @property
    def text(self):
        if self._text is None:
            self._text = self._text0 + "$"                           # csa/enhanced_fm_index.py:9
        return self._text

    @property
    def suffix_array(self):
        if self._sa is None:
            self._sa = _views.int_sequence(self._idx.sa)
        return self._sa

    @property
    def lcp_array(self):
        """LCP array of self.text in suffix-array order (no reference counterpart): lcp_array[0] = 0, lcp_array[r] =
        longest common prefix of the suffixes at suffix_array[r-1] and suffix_array[r].  Built on the device on
        first use."""
        if self._lcp is None:
            self._lcp = _views.int_sequence(self._idx.lcp())
        return self._lcp

    @property
    def bwt(self):
        if self._bwt is None:
            raw = self._E.to_host(self._idx.bwt).tobytes()
            self._bwt = self._smap.decode(raw) if self._str else raw
        return self._bwt

    @property
    def occ(self):
        if self._occ is None:
            self._occ = _views.occ_mapping(self._idx.wt)
            if self._str and not self._smap.identity:
                self._occ = {self._smap.symbol(ord(k)): v for k, v in self._occ.items()}
        return self._occ

    @property
    def device_index(self):
        return self._idx

    # ---- queries (:15-40)
    def find(self, query):
        l, r = self.find_range(query)
        if l == -1 or r == -1:
            return []
        E = self._E
        import torch
        rows = torch.arange(l, r + 1, dtype=torch.int32, device=self._idx.device)
        return self._idx.locate_rows(rows, use_samples=False).cpu().tolist()   # SA order, like :19

    def find_range(self, query):
        lo, hi = self.find_range_batch([query])
        return int(lo[0]), int(hi[0])

    def rank(self, character, index):
        """occ[character][index]; 0 for a symbol that never occurs; index clamped to n (:34-40)."""
        if isinstance(character, str) and self._smap is not None:
            enc = self._smap.encode(character)
            if enc is None or len(enc) != 1:
                return 0
            b = enc[0]
        else:
            b = ord(character) if isinstance(character, str) else int(character)
        if not 0 <= b < 256:
            return 0
        return int(self._idx.wt.rank(np.array([b], dtype=np.uint8), np.array([max(0, index)], dtype=np.int64)).item())

    # ---- batched additions
    def find_range_batch(self, queries):
        """Inclusive SA ranges for many patterns at once: (lo, hi) int64 numpy arrays; (-1, -1) = miss."""
        pat, off, absent = self._pack(queries)
        lo, hi = self._idx.count_batch(pat, off)
        lo, hi = self._E.to_host(lo), self._E.to_host(hi)
        if absent:                                   # a symbol the text cannot hold: (-1, -1) like :27-28
            lo[absent] = -1
            hi[absent] = -1
        return lo, hi

    def count_batch(self, queries):
        lo, hi = self.find_range_batch(queries)
        return np.where(lo >= 0, hi - lo + 1, 0)

    def find_batch(self, queries):
        """find() for many patterns: list of lists of positions, each in SA order."""
        pat, off, absent = self._pack(queries)
        o, p = self._idx.locate_batch(pat, off, use_samples=False)
        o, p = o.cpu().numpy(), p.cpu().numpy()
        gone = set(absent)
        return [[] if k in gone else p[o[k]:o[k + 1]].tolist() for k in range(len(o) - 1)]

    def _miss_pattern(self):
        """One byte the text does not hold (a search for it ends at once), b"" when all 256 occur."""
        plan = self._idx.wt.plan
        for b in range(255, -1, -1):
            if plan.code_of_sym[b] == 0xFFFF:
                return bytes([b])
        return b""

    def _pack(self, queries):
        """Patterns -> device CSR.  A str pattern holding a symbol the text's symbol map cannot express (a code point
        above 255 on latin-1 text, or one that never occurs in a re-coded text) is a miss by definition
        (csa/enhanced_fm_index.py:27-28: unseen symbol -> rank 0 -> (-1, -1)): it is searched as the one-symbol
        pattern of a byte the text does not hold, or overridden on the host when every byte occurs."""
        if self._smap is None or self._smap.identity:
            try:                                     # every pattern a latin-1 str: packed without a Python loop
                pat, off = self._E.pack_patterns(queries, self._idx.device)
                return pat, off, []
            except (TypeError, UnicodeEncodeError, ValueError):
                pass
        enc, absent = [], []
        for k, q in enumerate(queries):
            if isinstance(q, str):
                b = self._smap.encode(q) if self._smap is not None else q.encode("latin-1")
                if b is None:
                    absent.append(k)
                    b = self._miss_pattern()
                enc.append(b)
            else:
                enc.append(bytes(q))
        pat, off = self._E.pack_patterns(enc, self._idx.device)
        return pat, off, absent
