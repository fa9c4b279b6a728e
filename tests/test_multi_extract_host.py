"""CPU-only: the argument checks of the two extract entry points of the sliced index (hkcsa_multi_isa_samples,
hkcsa_multi_extract) run on the host before any CUDA call.  Every pointer below is a fake that is never
dereferenced: each call returns at a check."""
import ctypes as C

from hkcsa import _lib

FAKE = C.c_void_p(0x1000)


def _slice_plan(m, rate, marks):
    p = _lib.SsaPlan()
    assert _lib.load().hkcsa_ssa_plan_make_slice(m, rate, marks, C.byref(p)) == _lib.OK
    return p


def _isa(plans, lens, blobs=None, starts=None, out=FAKE):
    L = _lib.load()
    S = len(plans)
    k = max(S, 1)
    st = [0]
    for m in lens:
        st.append(st[-1] + m)
    st = st if starts is None else starts
    b = (C.c_void_p * k)(*([0x2000] * k if blobs is None else blobs))
    pl = (C.POINTER(_lib.SsaPlan) * k)(*[C.pointer(p) if p is not None else C.POINTER(_lib.SsaPlan)() for p in plans])
    return L.hkcsa_multi_isa_samples(S, b, pl, (C.c_uint64 * len(st))(*st), out, None)


def _err():
    return _lib.load().hkcsa_last_error()


def test_multi_isa_samples_argument_checks_without_gpu():
    # "banana$" cut into 4 + 3 rows at rate 2: marks 2 + 2 = ceil(7 / 2)
    good = [_slice_plan(4, 2, 2), _slice_plan(3, 2, 2)]
    other_rate = [_slice_plan(4, 2, 2), _slice_plan(3, 3, 2)]
    assert _isa(other_rate, [4, 3]) == _lib.EINVAL and b"rates" in _err()
    assert _isa([_slice_plan(4, 2, 2), _slice_plan(3, 2, 1)], [4, 3]) == _lib.EINVAL and b"add up" in _err()
    assert _isa([_slice_plan(4, 2, 3), _slice_plan(3, 2, 2)], [4, 3]) == _lib.EINVAL and b"add up" in _err()
    assert _isa(good, [4, 3], starts=[0, 5, 7]) == _lib.EINVAL and b"plan length" in _err()
    assert _isa(good, [4, 3], starts=[0, 4, 8]) == _lib.EINVAL and b"plan length" in _err()
    # ceil(n / rate) > 2^32: eight slices of 2^29 + 1 rows at rate 1 (plans widened by hand; never built)
    big = []
    for _ in range(8):
        p = _lib.SsaPlan.from_buffer_copy(bytes(_slice_plan(1000, 1, 1000)))
        p.n = p.n_samples = (1 << 29) + 1
        big.append(p)
    assert _isa(big, [p.n for p in big]) == _lib.ERANGE and b"2^32" in _err()
    assert _isa(good, [4, 3], starts=[0, 4, (1 << 40) + 1]) == _lib.ERANGE and b"2^40" in _err()
    # slice counts and null pointers
    assert _isa([], []) == _lib.EINVAL
    assert _isa(good * 5, [4, 3] * 5) == _lib.EINVAL and b"slices" in _err()
    assert _isa(good, [4, 3], out=None) == _lib.EINVAL
    assert _isa(good, [4, 3], blobs=[0x2000, 0]) == _lib.EINVAL and b"null" in _err()
    assert _isa([good[0], None], [4, 3]) == _lib.EINVAL and b"null" in _err()
    L = _lib.load()
    pl = (C.POINTER(_lib.SsaPlan) * 2)(*[C.pointer(p) for p in good])
    assert L.hkcsa_multi_isa_samples(2, None, pl, (C.c_uint64 * 3)(0, 4, 7), FAKE, None) == _lib.EINVAL
    assert L.hkcsa_multi_isa_samples(2, (C.c_void_p * 2)(0x2000, 0x2000), None, (C.c_uint64 * 3)(0, 4, 7), FAKE,
                                     None) == _lib.EINVAL
    # a rate of 0 in the first plan
    zero = [_lib.SsaPlan.from_buffer_copy(bytes(p)) for p in good]
    zero[0].rate = zero[1].rate = 0
    assert _isa(zero, [4, 3]) == _lib.EINVAL and b"rate" in _err()


def test_multi_extract_argument_checks_without_gpu():
    L = _lib.load()
    need = L.hkcsa_extract_scratch_bytes(3)

    def call(desc=FAKE, n=7, rate=2, isa=FAKE, R=3, begin=FAKE, out=FAKE, scratch=FAKE, nbytes=need):
        return L.hkcsa_multi_extract(desc, n, rate, isa, begin, FAKE, FAKE, R, out, scratch, nbytes, None)

    assert call(desc=None) == _lib.EINVAL
    assert call(isa=None) == _lib.EINVAL
    assert call(rate=0) == _lib.EINVAL
    assert call(n=0) == _lib.EINVAL
    assert call(n=(1 << 40) + 1) == _lib.ERANGE and b"2^40" in _err()
    assert call(begin=None) == _lib.EINVAL
    assert call(out=None) == _lib.EINVAL
    assert call(scratch=None) == _lib.EINVAL
    assert call(nbytes=need - 1) == _lib.ESCRATCH
    assert call(R=0, begin=None, out=None, scratch=None, nbytes=0) == _lib.OK     # nothing to do: no device work
