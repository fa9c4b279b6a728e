"""Drop-in for the reference's csa/csa.py on B200: ``FMIndex`` (:6-45 == main.py:6-46) with its
degenerate search kept as is, plus the ``CompressedSuffixArray(text, epsilon).locate(p)`` class
the reference's own benchmark imports but never defines (tests/benchmark.py:8,32,47), and a
``main()`` demo (:48-61).  The reference module cannot even be imported (it asks
csa.suffix_array for ``optimized_ksa``, :3); this one can.
"""
import math

import numpy as np

from csa.bwt import bwt_transform
from csa.suffix_array import build_suffix_array, optimized_ksa  # noqa: F401  (csa/csa.py:2-3)
from csa.wavelet_tree import WaveletTree
from hkcsa import views as _views


class FMIndex:
    """The reference's FMIndex: SA and BWT of the text WITHOUT a sentinel, per-symbol position
    lists, and a backward search that -- as written in the reference (:21-38) -- ends with
    (top, bottom) = (0, n-1) for every pattern, so find_pattern returns the whole suffix array."""

    def __init__(self, text):
        self.text = text
        self.suffix_array = build_suffix_array(text)          # :9
        self.bwt = bwt_transform(text, self.suffix_array)     # :10
        self.rank = self.precompute_rank()                    # :11

    def precompute_rank(self):
        """rank[c] = ascending positions of c in the BWT, keys in first-appearance order (:13-19).
        One stable counting-sort kernel (positions grouped by symbol)."""
        from hkcsa import engine
        n = len(self.bwt)
        if n == 0:
            return {}
        d_bwt = engine.to_device_u8(self.bwt)
        pos, start = engine.symbol_positions(d_bwt)
        first = {}
        present = [b for b in range(256) if start[b + 1] > start[b]]
        heads = pos.cpu().numpy() if n <= _views.MATERIALIZE_MAX else None
        for b in present:
            first[b] = int(heads[int(start[b])]) if heads is not None else int(pos[int(start[b])].item())
        rank = {}
        for b in sorted(present, key=lambda x: first[x]):
            s, e = int(start[b]), int(start[b + 1])
            if heads is not None:
                rank[chr(b)] = heads[s:e].tolist()
            else:
                rank[chr(b)] = _views.DeviceSequence(pos[s:e])
        return rank

    def backward_search(self, pattern):
        # The reference's loop (:21-38), restated: with n >= 1 the first iteration sets top = 0
        # ("top > 0" is false) and bottom = len(bwt) (or positions[n-1] = n-1 when the BWT is one
        # repeated symbol); later iterations keep that; the clamp gives (0, n-1).  An empty
        # pattern never enters the loop: also (0, n-1).  Empty text: range(0, 0).
        n = len(self.bwt)
        return list(range(0, n))

    def find_pattern(self, pattern):
        matches = self.backward_search(pattern)
        if isinstance(self.suffix_array, list):
            return [self.suffix_array[i] for i in matches if i < len(self.suffix_array)]
        return self.suffix_array.tolist()


class CompressedSuffixArray:
    """The index the reference's benchmark expects (tests/benchmark.py:25-52) and its README
    describes (README.md:4-11): text + '$', wavelet tree over the BWT for rank, and a suffix
    array sampled every s = ceil((log2 n)^epsilon) text positions, so ``locate`` walks at most
    s-1 LF steps per occurrence.  The full suffix array is dropped after sampling."""

    def __init__(self, text, epsilon=0.5, sa_sample_rate=None, entropy_orders=(), *, lcp=False):
        from hkcsa import engine
        self._E = engine
        self.text = text
        self.epsilon = epsilon
        self._is_str = isinstance(text, str)
        self._smap = engine.SymbolMap(text, extra="$") if self._is_str else None
        if self._smap is not None:
            d_text = engine.to_device_u8(self._smap.host_bytes(text), tail=self._smap.encode("$"))
            has_sentinel = "$" in text
        else:
            d_text = engine.to_device_u8(text, tail=b"$")
            has_sentinel = bool((d_text[:-1] == 0x24).any().item())
        n = d_text.numel()
        if sa_sample_rate is None:
            sa_sample_rate = max(1, math.ceil(max(1.0, math.log2(max(2, n))) ** epsilon))
        self.sa_sample_rate = int(sa_sample_rate)
        # A text that already holds '$' has no unique sentinel: suffix order is then not rotation order and LF walks
        # need not reach a sampled row.  Such an index keeps the full suffix array and locates through it (the
        # answers EnhancedFMIndex.find gives, csa/enhanced_fm_index.py:15-19) instead of through the samples.
        self.sentinel_unique = not has_sentinel
        self._idx = engine.DeviceIndex(d_text, sa_sample_rate=self.sa_sample_rate, keep_sa=True, keep_text=True)
        self.n = n
        # H_k of the indexed text (text + '$') for the requested orders, while the suffix array still exists
        self.entropy = {int(k): self._idx.entropy(int(k)) for k in entropy_orders}
        # lcp=True: Sadakane's 2n-bit encoding of the LCP array, built now because it needs the text and the full SA
        self.has_lcp = bool(lcp)
        if self.has_lcp:
            self._idx.build_lcp_bits()
        self._idx.text = None
        if not has_sentinel:
            self._idx.sa = None                                # the full suffix array is dropped after sampling

    @property
    def device_index(self):
        return self._idx

    @property
    def text(self):
        """The text the index was built from.  An index opened with load() holds no copy: the first access extracts
        it from the index."""
        if self._text is None:
            self._text = self.extract(0, self.n - 1)
        return self._text

    @text.setter
    def text(self, value):
        self._text = value

    def _pack(self, patterns):
        """Patterns -> device CSR; a str pattern with a symbol the text cannot hold becomes a pattern that misses."""
        enc = []
        for q in patterns:
            if isinstance(q, str):
                b = self._smap.encode(q) if self._smap is not None else q.encode("latin-1", "replace")
                if b is None:
                    b = self._miss_pattern()
                    if b is None:
                        raise ValueError("pattern holds a symbol outside the 256 byte symbols of the text")
                enc.append(b)
            else:
                enc.append(bytes(q))
        return self._E.pack_patterns(enc, self._idx.device)

    def _miss_pattern(self):
        plan = self._idx.wt.plan
        for b in range(255, -1, -1):
            if plan.code_of_sym[b] == 0xFFFF:
                return bytes([b])
        return None

    def count(self, pattern):
        return int(self.count_batch([pattern])[0])

    def locate(self, pattern):
        """Sorted text positions of every occurrence of `pattern`."""
        return self.locate_batch([pattern])[0]

    def count_batch(self, patterns):
        lo, hi = self._idx.count_batch(*self._pack(patterns))
        lo, hi = self._E.to_host(lo), self._E.to_host(hi)
        return np.where(lo >= 0, hi - lo + 1, 0)

    def locate_batch(self, patterns):
        off, pos = self._idx.locate_batch(*self._pack(patterns), use_samples=self.sentinel_unique)
        off, pos = off.cpu().numpy(), pos.cpu().numpy()
        return [sorted(pos[off[k]:off[k + 1]].tolist()) for k in range(len(off) - 1)]

    def lcp(self, rows):
        """LCP[rows] of the indexed text (text + '$') as an int64 numpy array: rows is an int or a sequence of suffix-
        array rows in [0, n); LCP[0] = 0, LCP[r] = longest common prefix of the suffixes in rows r-1 and r.  Answered
        from the 2n-bit encoding (needs lcp=True at construction) and a locate per row."""
        if not self.has_lcp:
            raise ValueError("this index holds no LCP encoding: build it with CompressedSuffixArray(..., lcp=True); "
                             "save() does not write the encoding, so an index opened with load() has none")
        import torch
        r = np.atleast_1d(np.asarray(rows, dtype=np.int64))
        if r.ndim != 1 or ((r < 0) | (r >= self.n)).any():
            raise ValueError(f"rows must lie in [0, n) with n = {self.n}")
        out = self._idx.lcp_rows(torch.from_numpy(r).to(self._idx.device), use_samples=self.sentinel_unique)
        return out.cpu().numpy().astype(np.int64)

    def space_report(self):
        """Index size next to the entropy bound: bits per symbol of the query blob and of the entropy-coded levels
        (what save(compressed=True) writes), the sampled SA, and n*H_k for the orders given at construction
        (README.md:4-11 of the reference: "space close to the k-th order entropy")."""
        rep = self._idx.space()
        rep["sa_sample_rate"] = self.sa_sample_rate
        rep["H_k_bits_per_symbol"] = dict(self.entropy)
        rep["n_H_k_bits"] = {k: v * self.n for k, v in self.entropy.items()}
        rep["coded_index_bits_per_symbol"] = rep["coded_level_bits_per_symbol"] + rep["sampled_sa_bits_per_symbol"]
        if self.has_lcp:
            rep["lcp_bits_per_symbol"] = self._idx._lcp_bits_held() / max(self.n, 1)
        return rep

    def extract(self, start, end):
        """text[start:end] from the index alone (Python slice semantics on the text without the sentinel): a str for a
        str text, bytes otherwise.  ValueError when the text held '$' in a way that keeps LF from inverting the suffix
        order (the index then cannot give the text back)."""
        return self.extract_batch([(start, end)])[0]

    def extract_batch(self, pairs):
        """[text[a:b] for (a, b) in pairs], every range extracted by one batched kernel call."""
        import torch
        m = self.n - 1
        bounds = np.array([slice(a, b).indices(m)[:2] for a, b in pairs], dtype=np.int64).reshape(-1, 2)
        bounds[:, 1] = np.maximum(bounds[:, 1], bounds[:, 0])           # a > b: the empty slice
        d = torch.from_numpy(bounds).to(self._idx.device)
        off, data = self._idx.extract_batch(d[:, 0], d[:, 1])
        off, data = off.cpu().numpy(), self._E.to_host(data).tobytes()
        if not self._is_str:
            return [data[off[k]:off[k + 1]] for k in range(len(bounds))]
        return [self._smap.decode(data[off[k]:off[k + 1]]) for k in range(len(bounds))]

    def save(self, path, compressed=True):
        """The index (DeviceIndex.save) plus what load() needs to answer as this object does: n, the sampling rate,
        epsilon, whether the sentinel was unique, str or bytes, the code points of a re-coded str alphabet and H_k."""
        back = self._smap.back if self._smap is not None else None
        meta = {"csa_meta": np.array([self.n, self.sa_sample_rate, int(self.sentinel_unique), int(self._is_str)],
                                     dtype=np.int64),
                "csa_epsilon": np.array([np.nan if self.epsilon is None else self.epsilon], dtype=np.float64),
                "csa_symbols": np.array([ord(c) for c in back] if back else [], dtype=np.int32),
                "csa_entropy": np.array(sorted(self.entropy.items()), dtype=np.float64).reshape(-1, 2)}
        self._idx.save(path, compressed=compressed, extra=meta)

    @classmethod
    def load(cls, path):
        """A query-only CompressedSuffixArray from a file save() wrote: count, locate, extract, space_report and
        index_bytes work; ``text`` is extracted from the index on first access."""
        from hkcsa import engine
        with np.load(path) as z:
            if "csa_meta" not in z.files:
                raise ValueError(f"{path} was not written by CompressedSuffixArray.save")
            n, rate, unique, is_str = (int(v) for v in z["csa_meta"])
            epsilon = float(z["csa_epsilon"][0])
            symbols = [chr(int(c)) for c in z["csa_symbols"]]
            entropy = {int(k): float(v) for k, v in z["csa_entropy"]}
        if not unique:
            raise ValueError("the saved text held the sentinel '$': such an index locates through its full suffix "
                             "array, which save() does not write")
        self = cls.__new__(cls)
        self._E = engine
        self._text = None
        self.epsilon = None if epsilon != epsilon else epsilon
        self._is_str = bool(is_str)
        self._smap = engine.SymbolMap.from_code_points(symbols) if self._is_str else None
        self.sa_sample_rate = rate
        self.sentinel_unique = True
        self._idx = engine.DeviceIndex.load(path)
        self.n = n
        self.entropy = entropy
        self.has_lcp = False
        return self

    def index_bytes(self):
        """Device bytes held by the index (wavelet tree blob + sampled SA blob [+ the suffix array, kept only when
        the text already holds the sentinel] [+ the LCP encoding, built with lcp=True])."""
        extra = self._idx.sa.numel() * 4 if self._idx.sa is not None else 0
        extra += self._idx._lcp_bits_held() // 8
        return int(self._idx.wt.blob.numel() + self._idx.ssa.blob.numel() + extra)


def main():
    text = "this is an example text"
    fm_index = FMIndex(text)
    pattern = "example"
    print(f"Searching for the pattern: '{pattern}'")
    matches = fm_index.find_pattern(pattern)
    print(f"Pattern '{pattern}' found at indices: {matches}")
    wavelet_tree = WaveletTree(text)
    compressed = wavelet_tree.compress()
    print(f"Wavelet Tree Compression: {compressed}")


if __name__ == "__main__":
    main()
