"""Long-pair batch alignment on the GPU (swb200_align_long_batch, swb200_batch_align_long, api.align_long_batch,
fasta.align_pairs): every pair gets exactly what api.align (swb200_align) returns for it alone, every score equals
swb200_score_long_batch's, pairs with a short side up to 1024 equal swb200_align_batch word for word, and the host,
device, chunked and two-GPU forms agree."""
import re

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import api, fasta, rng
from test_gpu_align_batch import _rescore

pytestmark = pytest.mark.gpu
PARAMS = (O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3))


def _ragged(seed, n, shorts=(), max_short=6000, max_long=20000):
    """Short sides 0 .. max_short, long sides up to max_long, planted and random, both orders."""
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    qs = list(shorts) + [int(r.integers(0, max_short + 1)) for _ in range(n - len(shorts))]
    for k, q in enumerate(qs):
        t = int(r.integers(q, max(q, min(max_long, 3 * q + 500)) + 1))
        a = rng.random_acgt(seed, 2 * k, t)
        if k % 2 == 0 and q > 4:
            o = int(r.integers(0, t - q + 1))
            b = rng.mutate(a[o:o + q], seed, 2 * k + 1, 0.08, 0.03)[:q]
        else:
            b = rng.random_acgt(seed, 2 * k + 1, q)
        pair = (bytes(b), bytes(a)) if k % 3 else (bytes(a), bytes(b))
        s1.append(pair[0]); s2.append(pair[1])
    return s1, s2


def _check_against_align(s1, s2, p, scores, spans, cigars, sample=None):
    for k in (range(len(s1)) if sample is None else sample):
        a, b = s1[k], s2[k]
        got = (int(scores[k]), tuple(int(x) for x in spans[k]), cigars[k])
        try:
            want = api.align(a, b, p)
        except api.SwbError as e:
            # gap_ext > gap_init: swb200_align merges two neighbouring opened gaps and refuses its own CIGAR; the batch
            # calls report them as two operations (include/swb200.h)
            assert p[3] > p[2] and "internal" in str(e)
            assert (got[0],) + got[1] == api.score_span(a, b, p)
            want = got
        assert got == want, (k, p, len(a), len(b), got[0], got[1], want[0], want[1])
        if got[0] > 0:
            assert _rescore(got[2], np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8), got[1], p) == (got[0], True)


EDGES = (1024, 1025, 255, 256, 257, 2049, 0, 6000)


@pytest.mark.parametrize("p", PARAMS)
def test_ragged_mix_equals_align(p):
    s1, s2 = _ragged(40 + PARAMS.index(p), 40, EDGES)
    s1.append(bytes(rng.random_acgt(41, 999, 1500))); s2.append(bytes(rng.random_acgt(41, 998, 20000)))
    scores, spans, cigars = api.align_long_batch(s1, s2, p)
    info = api.last_run()
    assert info["config"] == 320 and info["lanes"] == 32 and info["rows"] == 8 and info["bands"] == -(-6000 // 256)
    assert scores.tolist() == api.score_long_batch(s1, s2, p).tolist()
    _check_against_align(s1, s2, p, scores, spans, cigars)


def test_short_pairs_equal_align_batch():
    s1, s2 = _ragged(42, 300, (1024, 1, 0), max_short=1024, max_long=3000)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    for p in (O.DEFAULT, (2, -1, 1, 3)):
        want = api.align_batch_ops(f1, o1, l1, f2, o2, l2, p, 4096)
        got = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2, p, 4096)
        for w, g in zip(want, got):
            assert np.array_equal(w, g), p


def test_range_edge():
    a = b"A" * 32765
    assert api.align_long_batch([a], [a])[2] == ["32765="]
    x = rng.random_acgt(43, 0, 30000)
    y = rng.mutate(x, 43, 1, 0.08, 0.03)
    sc, sp, cg = api.align_long_batch([bytes(x)], [bytes(y)])
    assert (int(sc[0]), tuple(sp[0].tolist()), cg[0]) == api.align(bytes(x), bytes(y))
    with pytest.raises(api.SwbError) as e:
        api.align_long_batch([b"A" * 32766], [b"A" * 32766])
    assert e.value.code == -6


def _device_batch(torch, ctx, s1, s2, keep_order=False):
    dev = torch.device("cuda", 0)
    f1, o1, l1 = api._flatten(s1); f2, o2, l2 = api._flatten(s2)
    t = [torch.from_numpy(x).to(dev) for x in (f1, o1, l1, f2, o2, l2)]
    short, long_ = np.minimum(l1, l2), np.maximum(l1, l2)
    mx = (int(l1.max()), int(l2.max())) if keep_order else (int(short.max()), int(long_.max()))
    pb = api.PackedBatch(ctx, *[x.data_ptr() for x in t], len(s1), mx[0], mx[1], int((l1.astype(np.int64) * l2).sum()),
                         keep_order=keep_order)
    return pb, t


def test_call_forms_agree():
    import torch
    s1, s2 = _ragged(44, 160, EDGES, max_short=4000, max_long=9000)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    stride = 4096
    host = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2, O.DEFAULT, stride)
    ctx = api.Context(0)
    try:
        pb, keep = _device_batch(torch, ctx, s1, s2)
        n = len(s1)
        d = [torch.zeros(n, dtype=torch.int32, device="cuda:0"), torch.zeros((n, 4), dtype=torch.int32, device="cuda:0"),
             torch.zeros((n, stride), dtype=torch.int32, device="cuda:0"), torch.zeros(n, dtype=torch.int32, device="cuda:0")]
        pb.align_long(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), stride, d[3].data_ptr())
        dev_out = [x.cpu().numpy() for x in d]
        assert np.array_equal(dev_out[0], host[0]) and np.array_equal(dev_out[1], host[1])
        assert np.array_equal(dev_out[3], host[3]) and np.array_equal(dev_out[2].view(np.uint32), host[2])
        info = ctx.last_run()
        assert info["config"] == 320 and info["engine_launches"] == 2
        pb.close()
        pbk, keep2 = _device_batch(torch, ctx, s1, s2, keep_order=True)
        with pytest.raises(api.SwbError) as e:
            pbk.align_long(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), stride, d[3].data_ptr())
        assert e.value.code == -2
        pbk.close()
    finally:
        ctx.close()
    api.configure("batch_chunk_bytes", "200000")
    try:
        chunked = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2, O.DEFAULT, stride)
        assert all(np.array_equal(a, b) for a, b in zip(chunked, host))
        assert api.last_run()["aux_launches"] > 1
    finally:
        api.configure("batch_chunk_bytes", "0")


def test_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _ragged(45, 120, EDGES, max_short=4000, max_long=9000)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    one = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2)
    api.set_devices(2)
    try:
        two = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2)
    finally:
        api.set_devices(1)
    assert all(np.array_equal(a, b) for a, b in zip(one, two))


def test_ops_overflow_and_retry():
    s1, s2 = _ragged(46, 40, (1500, 3000), max_short=3000, max_long=6000)
    p = (2, -3, 5, 1)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    want = [api.align(a, b, p) for a, b in zip(s1, s2)]
    nops = [len(re.findall(r"\d+[=XID]", w[2])) for w in want]
    stride = int(np.median(nops))
    sc, sp, ops, cnt = api.align_long_batch_ops(f1, o1, l1, f2, o2, l2, p, stride)
    for k, w in enumerate(want):
        assert int(sc[k]) == w[0]
        if nops[k] > stride:
            assert cnt[k] == -nops[k] and not ops[k].any()
        else:
            assert api.cigar_string(ops[k, :cnt[k]]) == w[2]
    scores, spans, cigars = api.align_long_batch(s1, s2, p, ops_stride=stride)
    assert [(int(scores[k]), tuple(spans[k].tolist()), cigars[k]) for k in range(len(s1))] == want


def test_spans_larger_than_a_slot_take_pool_rounds():
    """400 planted 20 kb pairs: each span (202 MB of directions) is larger than a slot, and the pool (a fifth of free
    memory) cannot take them all in one round."""
    n = 400
    s1, s2 = [], []
    for k in range(n):
        x = rng.random_acgt(47, 2 * k, 20000)
        s1.append(bytes(x)); s2.append(bytes(rng.mutate(x, 47, 2 * k + 1, 0.05, 0.01)[:20000]))
    scores, spans, cigars = api.align_long_batch(s1, s2, ops_stride=8192)
    info = api.last_run()
    assert info["engine_launches"] > 2
    assert scores.tolist() == api.score_long_batch(s1, s2).tolist()
    _check_against_align(s1, s2, O.DEFAULT, scores, spans, cigars, sample=range(0, n, 40))


def test_fasta_routes_long_pairs_through_align_long(monkeypatch):
    r = np.random.default_rng(48)
    s1, s2 = [], []
    for k in range(96):
        if k % 3 == 0:                                           # reads against windows: the read batch
            w = rng.random_acgt(48, 2 * k, 800); s1.append(bytes(w[100:250])); s2.append(bytes(w))
        else:                                                    # 2-4 kb records: the long-pair batch
            a = rng.random_acgt(48, 2 * k, int(r.integers(2000, 4001)))
            b = rng.mutate(a, 48, 2 * k + 1, 0.08, 0.03) if k % 2 else rng.random_acgt(48, 2 * k + 1, int(r.integers(2000, 4001)))
            s1.append(bytes(a)); s2.append(bytes(b))
    ran = []
    orig = api.PackedBatch.align_long
    monkeypatch.setattr(api.PackedBatch, "align_long", lambda self, *a, **k: (ran.append(self.npairs), orig(self, *a, **k))[1])
    scores, spans, cigars = fasta.align_pairs(s1, s2)
    assert ran and ran[0] == 64
    want = [api.align(a, b) for a, b in zip(s1, s2)]
    assert [(int(scores[k]), tuple(spans[k].tolist()), cigars[k]) for k in range(len(s1))] == want
