"""Plain torch references for the succinct primitives under the index, exact and independent of libhkcsa (no `hkcsa`
import): the Golomb run code of a bit-vector, the size fields of its RRR class / offset code, and a vector that holds
every 15-bit block pattern once.  Rank and select are device_reference.bits_rank / bits_select.

Inputs are one byte per bit, any nonzero byte a one (what hkcsa_bitvec_build reads), on CPU or CUDA tensors.  Work
is chunked so that a vector of 2^30 bits fits beside its input: per chunk a few int64 temporaries, plus, for the Golomb
code, four int64 entries per run of ones and the output itself.  Pinned to the CPU oracle on small inputs by
tests/test_succinct_reference.py."""
from __future__ import annotations

import math

import torch

from device_reference import _chunks

CHUNK = 1 << 24          # bits per chunk
RRR_B = 15               # bits per block of the class / offset code
RRR_SB = 64              # blocks per superblock


# ------------------------------------------------------------------ runs of ones
def ones_runs(bits: torch.Tensor, chunk: int = CHUNK):
    """(start, length) int64 of every maximal run of ones, in order; the end of input closes the last run."""
    n = bits.numel()
    dev = bits.device
    starts, ends = [], []
    for a, b in _chunks(n, chunk):
        lo, hi = max(a - 1, 0), min(b + 1, n)
        w = torch.zeros(b - a + 2, dtype=torch.int8, device=dev)      # w[1 + i - a] = bit i, zero outside [0, n)
        w[1 + lo - a:1 + hi - a] = (bits[lo:hi] != 0).to(torch.int8)
        d = w[1:] - w[:-1]                                              # d[i - a] = bit i - bit (i - 1)
        starts.append(a + (d[:b - a] == 1).nonzero().flatten())
        ends.append(a + (d[1:] == -1).nonzero().flatten())              # bit i one, bit i + 1 zero: ends after i
    if not starts:
        z = torch.zeros(0, dtype=torch.int64, device=dev)
        return z, z
    s, e = torch.cat(starts), torch.cat(ends) + 1
    assert s.numel() == e.numel()
    return s, e - s


def golomb_encode(bits: torch.Tensor, m: int, chunk: int = CHUNK):
    """The Golomb-Rice run code of csrc/golomb.cu:1-7 -> (uint8 0/1 tensor, its length).  Every maximal run of ones of
    length v emits v // m zeros, a one, then v % m as exactly m bits, most significant first; runs of zeros emit
    nothing.  Runs come from the diff of the bits, each run's code is v // m + 1 + m bits long, and the code positions
    of every run follow from the exclusive prefix sum of those lengths: the output starts as zeros and only the
    terminating one and the remainder bits are written."""
    assert 1 <= m <= 62
    _, v = ones_runs(bits, chunk)
    q, r = v // m, v % m
    length = q + 1 + m
    off = torch.cumsum(length, 0) - length
    total = int(length.sum()) if v.numel() else 0
    out = torch.zeros(total, dtype=torch.uint8, device=bits.device)
    if total == 0:
        return out, 0
    head = off + q                                      # the one that ends the unary part
    out[head] = 1
    for b in range(m):
        out[head + 1 + b] = ((r >> (m - 1 - b)) & 1).to(torch.uint8)
    return out, total


# ------------------------------------------------------------------ RRR class / offset code
def rrr_class_widths() -> torch.Tensor:
    """ceil(log2 C(15, c)) for c = 0..15: the offset bits of a block of class c (int64[16])."""
    return torch.tensor([(math.comb(RRR_B, c) - 1).bit_length() for c in range(RRR_B + 1)], dtype=torch.int64)


def rrr_expected(bits: torch.Tensor, chunk: int = RRR_B * (1 << 20)) -> dict:
    """The size fields of the class / offset code of `bits`: nbits, nblocks = ceil(n / 15), nsuper = ceil(nblocks /
    64), ones, and stream_bits = the sum over 15-bit blocks (the last one zero-padded) of ceil(log2 C(15, popcount))."""
    assert chunk % RRR_B == 0
    n = bits.numel()
    nblocks = -(-n // RRR_B)
    width = rrr_class_widths().to(bits.device)
    ones = stream = 0
    for a, b in _chunks(n, chunk):
        x = (bits[a:b] != 0).to(torch.int64)
        pad = -(b - a) % RRR_B
        if pad:
            x = torch.cat([x, torch.zeros(pad, dtype=torch.int64, device=bits.device)])
        cls = x.view(-1, RRR_B).sum(1)
        ones += int(cls.sum())
        stream += int(width[cls].sum())
    return {"nbits": n, "nblocks": nblocks, "nsuper": -(-nblocks // RRR_SB), "ones": ones, "stream_bits": stream}


def all_patterns_vector(device=None) -> torch.Tensor:
    """32768 x 15 bits: block v holds the 15-bit value v, least significant bit first (the order in which rrr.cu:142
    reads a block).  Encoding it uses every entry of the pattern / offset_of tables once."""
    v = torch.arange(1 << RRR_B, dtype=torch.int64, device=device)
    return ((v[:, None] >> torch.arange(RRR_B, device=device)) & 1).to(torch.uint8).flatten()
