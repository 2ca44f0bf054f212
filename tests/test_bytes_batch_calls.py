"""The byte batch calls (swb200_score_batch_bytes, swb200_align_batch_bytes, swb200_batch_pack_device_bytes) without a
GPU: every bad call is refused before a device is touched, the limits are those of swb200_align_batch, and no byte value
is ever refused.  And fasta.plan_buckets' "bytes" bucket: exactly the non-ACGT pairs within the batch limits, and still
a partition of the pair ids."""
import ctypes as C

import numpy as np
import pytest

from concurrentproject_b200 import fasta

ARG, ALPHABET, RANGE = -2, -3, -6
LL, I, U, U8 = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_uint), C.POINTER(C.c_ubyte)


@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def _args(s1, s2, l1=None, o1=None):
    f1 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy()
    f2 = np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
    off = lambda s: np.concatenate([[0], np.cumsum([len(x) for x in s])[:-1]]).astype(np.int64)
    len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
    len2 = np.array([len(x) for x in s2], np.int32)
    off1 = np.array(o1, np.int64) if o1 is not None else off(s1)
    return f1, off1, len1, f2, off(s2), len2


def _score(lib, s1, s2, p=(1, -1, 1, 1), l1=None, o1=None, null_out=False, null_seq=False, n=None):
    from concurrentproject_b200 import _lib
    f1, o1, l1, f2, o2, l2 = _args(s1, s2, l1, o1)
    out = None if null_out else np.zeros(max(len(s1), 1), np.int32).ctypes.data_as(I)
    return lib.swb200_score_batch_bytes(None if null_seq else f1.ctypes.data_as(U8), o1.ctypes.data_as(LL), l1.ctypes.data_as(I),
                                        f2.ctypes.data_as(U8), o2.ctypes.data_as(LL), l2.ctypes.data_as(I),
                                        len(s1) if n is None else n, C.byref(_lib.Params(*p)), None, out)


def _align(lib, s1, s2, p=(1, -1, 1, 1), l1=None, o1=None, stride=8, null_out=False, null_seq=False, n=None):
    from concurrentproject_b200 import _lib
    f1, o1, l1, f2, o2, l2 = _args(s1, s2, l1, o1)
    k = max(len(s1), 1)
    sc, sp, ops, cnt = np.zeros(k, np.int32), np.zeros(4 * k, np.int32), np.zeros(k * max(stride, 1), np.uint32), np.zeros(k, np.int32)
    return lib.swb200_align_batch_bytes(None if null_seq else f1.ctypes.data_as(U8), o1.ctypes.data_as(LL), l1.ctypes.data_as(I),
                                        f2.ctypes.data_as(U8), o2.ctypes.data_as(LL), l2.ctypes.data_as(I),
                                        len(s1) if n is None else n, C.byref(_lib.Params(*p)), None, sc.ctypes.data_as(I),
                                        None if null_out else sp.ctypes.data_as(I), ops.ctypes.data_as(U), stride,
                                        cnt.ctypes.data_as(I))


@pytest.mark.parametrize("call", [_score, _align])
def test_bad_calls_are_refused_before_a_device_is_touched(lib, call):
    a, b = [b"ACGTN" * 30], [b"NNACGT" * 100]
    assert call(lib, a, b, null_out=True) == ARG
    assert call(lib, a, b, null_seq=True) == ARG
    assert call(lib, a, b, n=-1) == ARG
    assert call(lib, a, b, l1=[-5]) == ARG
    assert call(lib, a, b, o1=[-1]) == ARG
    for p in ((1, 1, 1, 1), (-1, -1, 1, 1), (1, -1, -1, 1), (1, -1, 1, 101), (100, -1, 28, 1)):
        assert call(lib, a, b, p=p) == ARG and b"limits" in lib.swb200_last_error(), p
    assert call(lib, [], []) == 0                                          # nothing to do
    if call is _align:
        assert call(lib, a, b, stride=0) == ARG                           # ops_stride < 1


@pytest.mark.parametrize("call", [_score, _align])
def test_limits_are_those_of_the_read_batch(lib, call):
    """min(len) > 1024: ARG; match * min(len) > 32766 - match: RANGE -- whatever the bytes."""
    assert call(lib, [b"N" * 1025], [b"n" * 1100]) == ARG and b"1024" in lib.swb200_last_error()
    assert call(lib, [b"ACGT" * 200, b"\x00" * 1025], [b"\xff" * 900, b"\x04" * 2000]) == ARG
    assert call(lib, [b"N" * 700], [b"X" * 800], p=(50, -1, 1, 1)) == RANGE
    assert call(lib, [b"\x00" * 1024], [b"\xff" * 1024], p=(32, -1, 1, 1)) == RANGE
    assert call(lib, [b"\x00" * 1024], [b"\xff" * 1024], p=(31, -1, 1, 1)) not in (ARG, RANGE, ALPHABET)


@pytest.mark.parametrize("call", [_score, _align])
def test_no_byte_value_is_refused(lib, call):
    """Every byte value, 0x00 and 0xFF included, in both sequences: never SWB200_ERR_ALPHABET (with a device the call
    succeeds; without one it fails at the device, after every check)."""
    every = bytes(range(256))
    s1 = [every[k:k + 40] for k in range(0, 256, 40)] + [b"acgtn", b"*-.", b""]
    s2 = [every[::-1][k:k + 60] for k in range(0, 256, 40)] + [b"ACGTN", b"", b"\x00"]
    rc = call(lib, s1, s2)
    assert rc != ALPHABET and rc not in (ARG, RANGE), rc


def test_device_pack_refuses_bad_arguments(lib):
    assert lib.swb200_batch_pack_device_bytes(None, None, None, None, None, None, None, 0, 0, 0, 0, None, None) == ARG
    assert lib.swb200_score_batch_bytes(None, None, None, None, None, None, 0, None, None, None) == 0
    assert lib.swb200_align_batch_bytes(None, None, None, None, None, None, 0, None, None, None, None, None, 1, None) == 0
    assert lib.swb200_align_batch_bytes(None, None, None, None, None, None, -1, None, None, None, None, None, 1, None) == ARG


def test_plan_buckets_bytes_bucket():
    r = np.random.default_rng(5)
    n = 4000
    l1 = r.integers(0, 3000, size=n)
    l2 = r.integers(0, 3000, size=n)
    ok = r.random(n) > 0.2
    short, long_ = np.minimum(l1, l2), np.maximum(l1, l2)
    for match in (1, 40):
        buckets = fasta.plan_buckets(l1, l2, ok, min_bucket=64, match=match)
        seen = np.concatenate([b.index for b in buckets])
        assert sorted(seen.tolist()) == list(range(n))                       # a partition of the pair ids
        eligible = ~ok & (short <= fasta.BATCH_MAX_SHORT) & (match * short <= 32766 - match)
        by = [b for b in buckets if b.kind == "bytes"]
        assert len(by) == 1 and sorted(by[0].index.tolist()) == np.flatnonzero(eligible).tolist()
        assert (np.diff(long_[by[0].index]) <= 0).all()                     # longest first
        single = np.concatenate([b.index for b in buckets if b.kind == "single"])
        assert not eligible[single].any()
        assert ((short[single] > fasta.BATCH_MAX_SHORT) | (match * short[single] > 32766 - match)).all()
    # all pairs ACGT: no bytes bucket
    assert not [b for b in fasta.plan_buckets(l1, l2, np.ones(n, bool), min_bucket=64) if b.kind == "bytes"]
