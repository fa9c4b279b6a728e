"""Exact LCP array for the LCP tests: Kasai's algorithm (tests/lcp_kasai.c), independent of libhkcsa.

The C source is compiled on first use into the system's temporary directory (the repository tree may be read-only
where the tests run), under a name that carries a hash of the source, and loaded with ctypes.  O(n) time and 4n bytes
beside its inputs: seconds at n = 2^30 on one host core.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lcp_kasai.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"hkcsa_lcp_kasai_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or shutil.which("cc"))
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(so))
            os.close(fd)
            subprocess.check_call([cc, "-O2", "-fPIC", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)                  # atomic: concurrent test processes never load a half-written file
        L = C.CDLL(so)
        L.lcp_kasai.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.lcp_kasai.restype = C.c_int
        _lib = L
    return _lib


def lcp_kasai(text, sa) -> np.ndarray:
    """LCP array in suffix-array order: lcp[0] = 0, lcp[r] = longest common prefix of the suffixes sa[r-1] and sa[r].
    text: bytes or a uint8 array; sa: any valid suffix array of it."""
    t = np.frombuffer(bytes(text), dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else \
        np.ascontiguousarray(text, dtype=np.uint8)
    sa = np.ascontiguousarray(sa, dtype=np.uint32)
    if len(sa) != len(t):
        raise ValueError("the suffix array must have one entry per text symbol")
    out = np.zeros(len(t), dtype=np.uint32)
    if len(t) and _load().lcp_kasai(t.ctypes.data, len(t), sa.ctypes.data, out.ctypes.data):
        raise MemoryError("lcp_kasai: out of host memory")
    return out
