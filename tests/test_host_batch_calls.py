"""The host batch calls (swb200_score_batch, swb200_score_banded_batch, swb200_score_batch_packed,
swb200_score_banded_batch_packed, swb200_align_batch) share one length scan, one stride rule, one sharding path and one
copy/pack pipeline.  Without a GPU: every call refuses bad input before it touches a device, and the strides of the
resident 2-bit layout follow the documented formula.  On the GPU: the alignment host call over many small chunks, and
the sharded calls' run info and kernel choice."""
import ctypes as C
import shutil

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

ARG, RANGE = -2, -6
needs_nvcc = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")
LL, I, U64 = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)
U8 = C.POINTER(C.c_ubyte)


@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def _ascii(s1, s2, l1=None, o1=None):
    """Flattened host arrays of a pair list; l1 / o1 replace seq1's lengths / offsets."""
    f1 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy()
    f2 = np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
    off = lambda s: np.concatenate([[0], np.cumsum([len(x) for x in s])[:-1]]).astype(np.int64)
    len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
    len2 = np.array([len(x) for x in s2], np.int32)
    off1 = np.array(o1, np.int64) if o1 is not None else off(s1)
    return f1, off1, len1, f2, off(s2), len2


def _params(p):
    from concurrentproject_b200 import _lib
    return C.byref(_lib.Params(*p))


def _score_ascii(lib, s1, s2, p=(1, -1, 1, 1), band=None, l1=None, o1=None, null_out=False, n=None):
    f1, o1, l1, f2, o2, l2 = _ascii(s1, s2, l1, o1)
    n = len(s1) if n is None else n
    out = None if null_out else np.zeros(max(len(s1), 1), np.int32).ctypes.data_as(I)
    args = (f1.ctypes.data_as(U8), o1.ctypes.data_as(LL), l1.ctypes.data_as(I), f2.ctypes.data_as(U8), o2.ctypes.data_as(LL),
            l2.ctypes.data_as(I), n)
    if band is None:
        return lib.swb200_score_batch(*args, _params(p), None, out)
    return lib.swb200_score_banded_batch(*args, band[0], band[1], _params(p), None, out)


def _score_packed(lib, ql, tl, p=(1, -1, 1, 1), band=None, strides=None, null_out=False, n=None):
    ql, tl = np.array(ql, np.int32), np.array(tl, np.int32)
    if strides is None:
        mq, mt = int(max(ql.max(), 0)), int(max(tl.max(), 0))
        extra = 2 if band is not None else 0
        strides = (max(1, (mq + 31) // 32) + extra, max(1, (mt + 31) // 32) + 2)
    qw = np.zeros(len(ql) * strides[0] + 1, np.uint64)
    tw = np.zeros(len(ql) * strides[1] + 1, np.uint64)
    n = len(ql) if n is None else n
    out = None if null_out else np.zeros(max(len(ql), 1), np.int32).ctypes.data_as(I)
    args = (qw.ctypes.data_as(U64), strides[0], tw.ctypes.data_as(U64), strides[1], ql.ctypes.data_as(I), tl.ctypes.data_as(I), n)
    if band is None:
        return lib.swb200_score_batch_packed(*args, _params(p), None, out)
    return lib.swb200_score_banded_batch_packed(*args, band[0], band[1], _params(p), None, out)


@needs_nvcc
def test_ascii_score_batches_refuse_bad_input_without_a_gpu(lib):
    ok = ([b"ACGT", b"AC"], [b"ACGTT", b"CA"])
    for band in (None, (-32, 31)):
        assert _score_ascii(lib, *ok, band=band, null_out=True) == ARG                    # null output
        assert _score_ascii(lib, *ok, band=band, n=-1) == ARG
        assert _score_ascii(lib, [], [], band=band) == 0                                   # nothing to do
        null = (None,) * 6
        if band is None:
            assert lib.swb200_score_batch(*null, 0, None, None, None) == 0
        else:
            assert lib.swb200_score_banded_batch(*null, 0, -32, 31, None, None, None) == 0
        assert _score_ascii(lib, *ok, band=band, l1=[4, -1]) == ARG                        # negative length
        assert _score_ascii(lib, *ok, band=band, o1=[0, -2]) == ARG                        # negative offset
        assert _score_ascii(lib, *ok, band=band, p=(1, 1, 1, 1)) == ARG                    # parameters outside the limits
        assert b"limits" in lib.swb200_last_error()
        long_pair = ([b"A" * 700, b"AC"], [b"C" * 800, b"CA"])
        assert _score_ascii(lib, *long_pair, band=band, p=(50, -1, 1, 1)) == RANGE         # match * min(len) > 32766 - match
    assert _score_ascii(lib, [b"A" * 1025], [b"C" * 1100]) == ARG                          # short side over 1024
    assert b"1024" in lib.swb200_last_error()
    assert _score_ascii(lib, *ok, band=(-32, 40)) == ARG                                   # not 64 diagonals
    seq = lambda b: C.cast(C.c_char_p(b), U8)
    assert lib.swb200_score_banded(seq(b"ACGT"), 4, seq(b"ACGT"), 4, -32, 40, None, C.byref(C.c_int())) == ARG
    assert lib.swb200_score_banded(seq(b"A" * 700), 700, seq(b"C" * 800), 800, -32, 31, _params((50, -1, 1, 1)),
                                   C.byref(C.c_int())) == RANGE


@needs_nvcc
def test_packed_score_batches_refuse_bad_input_without_a_gpu(lib):
    ok = ([4, 2], [5, 2])
    for band in (None, (-32, 31)):
        assert _score_packed(lib, *ok, band=band, null_out=True) == ARG                    # null output
        assert _score_packed(lib, *ok, band=band, n=-1) == ARG
        assert _score_packed(lib, [0], [0], band=band, n=0) == 0                            # nothing to do
        assert _score_packed(lib, [4, -1], [5, 2], band=band) == ARG                       # negative length
        assert _score_packed(lib, *ok, band=band, p=(1, 1, 1, 1)) == ARG                   # parameters outside the limits
        assert _score_packed(lib, [700, 2], [800, 2], band=band, p=(50, -1, 1, 1)) == RANGE
        small = (1, 3) if band is None else (3, 3)                                         # strides of 32-symbol pairs
        assert _score_packed(lib, [33, 2], [33, 2], band=band, strides=small) == ARG       # q does not fit
        assert _score_packed(lib, [2, 2], [33, 2], band=band, strides=small) == ARG        # t does not fit
    assert _score_packed(lib, [1025], [1100]) == ARG                                       # short side over 1024
    assert _score_packed(lib, [5], [4]) == ARG                                             # q longer than t
    assert _score_packed(lib, *ok, band=(-32, 40)) == ARG                                  # not 64 diagonals
    assert _score_packed(lib, *ok, strides=(0, 3)) == ARG and _score_packed(lib, *ok, band=(-32, 31), strides=(2, 3)) == ARG


@needs_nvcc
def test_strides_follow_the_layout(lib):
    """One word per 32 symbols, at least one; +2 words on the streamed side (the kernels prefetch one word past the end),
    +2 on both sides of a banded batch."""
    from concurrentproject_b200 import api
    words = lambda n: max(1, (n + 31) // 32)
    for short, long_ in ((0, 0), (0, 31), (31, 32), (32, 33), (33, 1024), (1024, 1024), (1024, 70000)):
        assert api.batch_strides(short, long_) == (words(short), words(long_) + 2)
    for l1, l2 in ((0, 0), (31, 32), (33, 1024), (1024, 31)):
        s1, s2 = [b"A" * l1, b"C"], [b"G" * l2, b"T"]
        f1, o1, n1, f2, o2, n2 = _ascii(s1, s2)
        _, st1, _, st2 = api.pack_banded_host(f1, o1, n1, f2, o2, n2)
        assert (st1, st2) == (words(max(l1, 1)) + 2, words(max(l2, 1)) + 2)


def _ragged(seed, n, short_lo, short_hi, long_hi):
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(n):
        a = rng.random_acgt(seed, k, int(r.integers(short_lo, short_hi + 1)))
        b = rng.mutate(a, seed, 1000 + k, 0.06, 0.02) if k % 2 else rng.random_acgt(seed, 5000 + k, int(r.integers(len(a), long_hi + 1)))
        s1.append(bytes(a)); s2.append(bytes(b))
    return s1, s2


@pytest.mark.gpu
def test_align_batch_in_many_chunks_equals_one_chunk():
    """The alignment host call over the shared copy/pack pipeline, cut into dozens of chunks, pairs in non-monotone
    offset order."""
    from concurrentproject_b200 import api
    s1, s2 = _ragged(41, 500, 0, 300, 1000)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    perm = np.random.default_rng(2).permutation(len(s1))
    o1, l1, o2, l2 = o1[perm].copy(), l1[perm].copy(), o2[perm].copy(), l2[perm].copy()
    p = (2, -3, 5, 1)
    want = api.align_batch_ops(f1, o1, l1, f2, o2, l2, p)
    api.configure("batch_chunk_bytes", "20000")
    try:
        got = api.align_batch_ops(f1, o1, l1, f2, o2, l2, p)
        info = api.last_run()
    finally:
        api.configure("batch_chunk_bytes", "0")
    assert info["aux_launches"] >= 10
    for w, g in zip(want, got):
        assert np.array_equal(w, g)
    assert np.array_equal(want[0], O.gotoh_batch([s1[k] for k in perm], [s2[k] for k in perm], p))


def _need_two_gpus():
    from concurrentproject_b200 import _lib
    if _lib.load().swb200_device_count() < 2:
        pytest.skip("needs two GPUs")


@pytest.mark.gpu
def test_sharded_packed_call_sums_launches_over_gpus():
    from concurrentproject_b200 import api
    _need_two_gpus()
    s1, s2 = _ragged(42, 400, 1, 150, 700)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    qw, qs, tw, ts, ql, tl = api.pack_batch_host(f1, o1, l1, f2, o2, l2)
    half = (len(s1) + 1) // 2
    api.configure("batch_chunk_bytes", "4000")
    try:
        alone = []
        for k0, k1 in ((0, half), (half, len(s1))):
            got = api.score_batch_packed(qw[k0 * qs:k1 * qs], qs, tw[k0 * ts:k1 * ts], ts, ql[k0:k1], tl[k0:k1])
            assert np.array_equal(got, O.gotoh_batch(s1[k0:k1], s2[k0:k1]))
            alone.append(api.last_run()["engine_launches"])
        api.set_devices(2)
        try:
            both = api.score_batch_packed(qw, qs, tw, ts, ql, tl)
            info = api.last_run()
        finally:
            api.set_devices(1)
    finally:
        api.configure("batch_chunk_bytes", "0")
    assert np.array_equal(both, O.gotoh_batch(s1, s2))
    assert min(alone) > 1 and info["engine_launches"] == sum(alone), (alone, info)


@pytest.mark.gpu
def test_sharded_ascii_batch_with_halves_of_different_size_classes():
    """Every range of a sharded call runs the kernel the whole batch's longest short side needs."""
    from concurrentproject_b200 import api
    _need_two_gpus()
    a1, a2 = _ragged(43, 100, 1, 128, 400)
    b1, b2 = _ragged(44, 100, 600, 700, 900)
    s1, s2 = a1 + b1, a2 + b2
    api.set_devices(2)
    try:
        got = api.score_batch(s1, s2)
    finally:
        api.set_devices(1)
    assert np.array_equal(got, O.gotoh_batch(s1, s2))
