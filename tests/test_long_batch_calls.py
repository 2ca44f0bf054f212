"""The multi-band batch calls (swb200_score_long_batch, swb200_batch_score_long) without a GPU: every bad call is refused
before a device is touched.  And fasta.plan_buckets' "long" bucket: exactly the eligible pairs, only when the batch
beats one single-pair call per pair, and still a partition of the pair ids."""
import ctypes as C

import numpy as np
import pytest

from concurrentproject_b200 import fasta

ARG, RANGE = -2, -6
LL, I, U8 = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_ubyte)


@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def _call(lib, s1, s2, p=(1, -1, 1, 1), rows=0, l1=None, o1=None, null_out=False, null_seq=False, n=None):
    from concurrentproject_b200 import _lib
    f1 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy()
    f2 = np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
    off = lambda s: np.concatenate([[0], np.cumsum([len(x) for x in s])[:-1]]).astype(np.int64)
    len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
    len2 = np.array([len(x) for x in s2], np.int32)
    off1 = np.array(o1, np.int64) if o1 is not None else off(s1)
    off2 = off(s2)
    out = None if null_out else np.zeros(max(len(s1), 1), np.int32).ctypes.data_as(I)
    o = _lib.Options(); o.rows = rows
    return lib.swb200_score_long_batch(None if null_seq else f1.ctypes.data_as(U8), off1.ctypes.data_as(LL),
                                       len1.ctypes.data_as(I), f2.ctypes.data_as(U8), off2.ctypes.data_as(LL),
                                       len2.ctypes.data_as(I), len(s1) if n is None else n,
                                       C.byref(_lib.Params(*p)), C.byref(o), out)


def test_bad_calls_are_refused_before_a_device_is_touched(lib):
    a, b = [b"ACGT" * 400], [b"ACGT" * 600]
    assert _call(lib, a, b, null_out=True) == ARG
    assert _call(lib, a, b, null_seq=True) == ARG
    assert _call(lib, a, b, n=-1) == ARG
    assert _call(lib, a, b, l1=[-5]) == ARG
    assert _call(lib, a, b, o1=[-1]) == ARG
    for rows in (1, 3, 5, 14, 17, -2):
        assert _call(lib, a, b, rows=rows) == ARG, rows
    # the 16-bit range: match * min(len) <= 32766 - match
    big = [b"A" * 32766]
    assert _call(lib, big, big) == RANGE
    assert _call(lib, [b"A" * 9000], [b"A" * 9000], p=(4, -1, 1, 1)) == RANGE
    assert lib.swb200_batch_score_long(None, None, None, None, None) == ARG
    assert _call(lib, [], []) == 0                                         # nothing to do


def test_plan_buckets_long_bucket():
    r = np.random.default_rng(3)
    n = 3000
    l1 = r.integers(0, 6000, size=n)
    l2 = r.integers(0, 6000, size=n)
    ok = r.random(n) > 0.05
    short, long_ = np.minimum(l1, l2), np.maximum(l1, l2)
    for match in (1, 8):
        buckets = fasta.plan_buckets(l1, l2, ok, min_bucket=64, match=match)
        seen = np.concatenate([b.index for b in buckets])
        assert sorted(seen.tolist()) == list(range(n))                       # a partition of the pair ids
        eligible = ok & (short > fasta.BATCH_MAX_SHORT) & (match * short <= 32766 - match)
        lng = [b for b in buckets if b.kind == "long"]
        assert len(lng) == 1 and sorted(lng[0].index.tolist()) == np.flatnonzero(eligible).tolist()
        idx = lng[0].index
        padded = -(-short[idx] // 1024) * 1024 * (long_[idx] + 63)
        assert (np.diff(padded) <= 0).all()                                  # largest padded area first
        single = np.concatenate([b.index for b in buckets if b.kind == "single"])
        assert (~ok[single] | (short[single] > fasta.BATCH_MAX_SHORT)).all()
        assert not eligible[single].any()
    # few long pairs: the single-pair engine is faster (measured crossover, fasta.long_batch_pays), so they stay there
    few_l1 = np.array([20000] * 3 + [100])
    few = fasta.plan_buckets(few_l1, few_l1 + 5, np.ones(4, bool), min_bucket=1)
    assert not [b for b in few if b.kind == "long"]
    assert sorted(next(b for b in few if b.kind == "single").index.tolist()) == [0, 1, 2]
    many_l1 = np.array([20000] * 300 + [100])
    many = fasta.plan_buckets(many_l1, many_l1 + 5, np.ones(301, bool), min_bucket=1)
    assert sorted(next(b for b in many if b.kind == "long").index.tolist()) == list(range(300))
    assert not [b for b in many if b.kind == "single"]


def test_cost_model_follows_the_measured_crossover():
    """Each (length, count) point of the recorded crossover: the router picks the multi-band call exactly where it was
    measured faster than one single-pair call per pair."""
    import json
    from pathlib import Path
    rec = json.loads((Path(__file__).resolve().parent.parent / "profiles" / "r06_long_batch.json").read_text())
    for c in rec["crossover"]:
        n, L = c["pairs"], c["length"]
        assert fasta.long_batch_pays(np.full(n, L), np.full(n, L)) == (c["batch_s"] < c["loop_s_est"]), c
