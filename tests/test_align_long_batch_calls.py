"""The long-pair batch alignment calls (swb200_align_long_batch, swb200_batch_align_long) without a GPU: every bad call
is refused before a device is touched.  And fasta.plan_buckets with the alignment cost model: a partition of the pair
ids whose "long" bucket follows align_long_batch_pays, while the default routing stays long_batch_pays'."""
import ctypes as C

import numpy as np
import pytest

from concurrentproject_b200 import fasta

ARG, RANGE, ALPHABET = -2, -6, -3
LL, I, U8, U = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_ubyte), C.POINTER(C.c_uint)


@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def _call(lib, s1, s2, p=(1, -1, 1, 1), stride=8, l1=None, o1=None, null_out=False, null_seq=False, n=None):
    from concurrentproject_b200 import _lib
    f1 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy()
    f2 = np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
    off = lambda s: np.concatenate([[0], np.cumsum([len(x) for x in s])[:-1]]).astype(np.int64)
    len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
    len2 = np.array([len(x) for x in s2], np.int32)
    off1 = np.array(o1, np.int64) if o1 is not None else off(s1)
    off2 = off(s2)
    k = max(len(s1), 1)
    sc, sp, ops, cnt = np.zeros(k, np.int32), np.zeros(4 * k, np.int32), np.zeros(k * max(stride, 1), np.uint32), np.zeros(k, np.int32)
    return lib.swb200_align_long_batch(None if null_seq else f1.ctypes.data_as(U8), off1.ctypes.data_as(LL),
                                       len1.ctypes.data_as(I), f2.ctypes.data_as(U8), off2.ctypes.data_as(LL),
                                       len2.ctypes.data_as(I), len(s1) if n is None else n, C.byref(_lib.Params(*p)), None,
                                       sc.ctypes.data_as(I), None if null_out else sp.ctypes.data_as(I),
                                       ops.ctypes.data_as(U), stride, cnt.ctypes.data_as(I))


def test_bad_calls_are_refused_before_a_device_is_touched(lib):
    a, b = [b"ACGT" * 400], [b"ACGT" * 600]
    assert _call(lib, a, b, null_out=True) == ARG
    assert _call(lib, a, b, null_seq=True) == ARG
    assert _call(lib, a, b, n=-1) == ARG
    assert _call(lib, a, b, stride=0) == ARG
    assert _call(lib, a, b, l1=[-5]) == ARG
    assert _call(lib, a, b, o1=[-1]) == ARG
    assert _call(lib, a, b, p=(1, 1, 1, 1)) == ARG                          # a positive mismatch
    assert _call(lib, a, b, p=(1, -1, -1, 1)) == ARG                        # a negative gap cost
    # the range of swb200_score_long_batch: match * min(len) <= 32766 - match, whatever the longer side
    big = [b"A" * 32766]
    assert _call(lib, big, big) == RANGE
    assert _call(lib, [b"A" * 9000], [b"A" * 9000], p=(4, -1, 1, 1)) == RANGE
    assert _call(lib, [b"A" * 700], [b"C" * 800], p=(50, -1, 1, 1)) == RANGE
    assert lib.swb200_batch_align_long(None, None, None, None, None, None, None, 8, None) == ARG
    assert lib.swb200_align_long_batch(None, None, None, None, None, None, 0, None, None, None, None, None, 1, None) == 0
    assert lib.swb200_align_long_batch(None, None, None, None, None, None, -1, None, None, None, None, None, 1, None) == ARG


def test_plan_buckets_with_the_alignment_cost_model():
    r = np.random.default_rng(5)
    n = 3000
    l1 = r.integers(0, 6000, size=n)
    l2 = r.integers(0, 6000, size=n)
    ok = r.random(n) > 0.05
    short, long_ = np.minimum(l1, l2), np.maximum(l1, l2)
    eligible = ok & (short > fasta.BATCH_MAX_SHORT) & (short <= 32765)
    default = fasta.plan_buckets(l1, l2, ok, min_bucket=64)
    aligned = fasta.plan_buckets(l1, l2, ok, min_bucket=64, pays=fasta.align_long_batch_pays)
    for buckets in (default, aligned):
        assert sorted(np.concatenate([b.index for b in buckets]).tolist()) == list(range(n))
        lng = [b for b in buckets if b.kind == "long"]
        assert len(lng) == 1 and sorted(lng[0].index.tolist()) == np.flatnonzero(eligible).tolist()
    # the read batch buckets do not depend on the cost model
    rb = lambda bs: [(b.cap, b.index.tolist()) for b in bs if b.kind == "batch"]
    assert rb(default) == rb(aligned)
    # the default routing is the scoring one: same buckets as before the keyword existed
    assert [(b.kind, b.cap, b.index.tolist()) for b in default] == \
        [(b.kind, b.cap, b.index.tolist()) for b in fasta.plan_buckets(l1, l2, ok, min_bucket=64, pays=fasta.long_batch_pays)]
    # a cost model that never pays sends every long pair to the single-pair engine
    none = fasta.plan_buckets(l1, l2, ok, min_bucket=64, pays=lambda s, l: False)
    assert not [b for b in none if b.kind == "long"]
    single = np.concatenate([b.index for b in none if b.kind == "single"])
    assert eligible[single].sum() == eligible.sum()


def test_alignment_cost_model_follows_the_measured_crossover():
    """Each (length, count) point of the recorded crossover: the router picks the long-pair alignment call exactly where
    it was measured faster than one swb200_align_device call per pair."""
    import json
    from pathlib import Path
    rec = json.loads((Path(__file__).resolve().parent.parent / "profiles" / "r07_align_long_batch.json").read_text())
    assert rec["crossover"]
    for c in rec["crossover"]:
        n, L = c["pairs"], c["length"]
        assert fasta.align_long_batch_pays(np.full(n, L), np.full(n, L)) == (c["batch_s"] < c["loop_s_est"]), c
