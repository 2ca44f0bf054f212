"""The multi-band batch calls on the GPU: every score equals the single-pair engine's (swb200_score_ex) for ragged pairs
with short sides up to 6 000 and long sides up to 20 000, and the C oracle on a subset; short pairs give exactly
swb200_score_batch's scores for every R; the 16-bit range edge; host, device-resident, chunked and two-GPU forms agree;
fasta routes long pairs through the "long" bucket."""
import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import api, fasta, rng

pytestmark = pytest.mark.gpu
PARAMS = (O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (1, -1, 2, 1), (2, -1, 1, 3))


def _ragged(seed, n, shorts=(), max_short=6000, max_long=20000):
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
        pair = (bytes(b), bytes(a)) if k % 3 else (bytes(a), bytes(b))          # both orders
        s1.append(pair[0]); s2.append(pair[1])
    return s1, s2


EDGES = (1024, 1025, 2048, 2049, 3071, 0, 6000)


def test_ragged_mix_equals_single_pair_engine():
    s1, s2 = _ragged(11, 60, EDGES)
    s1.append(bytes(rng.random_acgt(11, 999, 1500))); s2.append(bytes(rng.random_acgt(11, 998, 20000)))
    for p in PARAMS:
        got = api.score_long_batch(s1, s2, p)
        want = [api.score(a, b, p) for a, b in zip(s1, s2)]
        assert got.tolist() == want, p
    sub1, sub2 = s1[:12], s2[:12]
    assert api.score_long_batch(sub1, sub2).tolist() == O.gotoh_batch(sub1, sub2).tolist()
    info = api.last_run()
    assert info["config"] == 332 and info["rows"] == 16 and info["bands"] == -(-max(map(min, map(len, sub1), map(len, sub2))) // 1024)


def test_short_pairs_equal_the_batch_kernel():
    s1, s2 = _ragged(12, 300, (1024, 1, 0), max_short=1024, max_long=3000)
    for p in (O.DEFAULT, (2, -3, 5, 1)):
        want = api.score_batch(s1, s2, p).tolist()
        for rows in (2, 4, 16, 0):
            assert api.score_long_batch(s1, s2, p, rows=rows).tolist() == want, (p, rows)
            assert api.last_run()["bands"] == -(-1024 // (64 * (rows or 16)))
        assert api.score_long_batch(s1, s2, p, no_linear=True).tolist() == want


def test_range_edge():
    a = b"A" * 32765
    assert api.score_long_batch([a], [a]).tolist() == [32765]
    x = rng.random_acgt(13, 0, 30000)
    y = rng.mutate(x, 13, 1, 0.08, 0.03)
    assert api.score_long_batch([bytes(x)], [bytes(y)]).tolist() == [api.score(x, y)]
    with pytest.raises(api.SwbError):
        api.score_long_batch([b"A" * 32766], [b"A" * 32766])


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
    s1, s2 = _ragged(14, 200, EDGES, max_short=4000, max_long=9000)
    host = api.score_long_batch(s1, s2)
    ctx = api.Context(0)
    try:
        pb, keep = _device_batch(torch, ctx, s1, s2)
        d = torch.empty(len(s1), dtype=torch.int32, device="cuda:0")
        for p in (O.DEFAULT, (2, -3, 5, 1)):
            pb.score_long(d.data_ptr(), p)
            assert d.cpu().numpy().tolist() == api.score_long_batch(s1, s2, p).tolist(), p
        pb.score_long(d.data_ptr())
        assert d.cpu().numpy().tolist() == host.tolist()
        info = ctx.last_run()
        assert info["config"] == 332 and info["engine_launches"] == 1 and info["bands"] == 6
        pb.close()
        pbk, keep2 = _device_batch(torch, ctx, s1, s2, keep_order=True)
        with pytest.raises(api.SwbError) as e:
            pbk.score_long(d.data_ptr())
        assert e.value.code == -2
        pbk.close()
    finally:
        ctx.close()
    api.configure("batch_chunk_bytes", "200000")
    try:
        assert api.score_long_batch(s1, s2).tolist() == host.tolist()
        info = api.last_run()
        assert info["engine_launches"] == info["aux_launches"] > 1
    finally:
        api.configure("batch_chunk_bytes", "0")


def test_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _ragged(15, 120, EDGES, max_short=4000, max_long=9000)
    one = api.score_long_batch(s1, s2)
    api.set_devices(2)
    try:
        assert api.score_long_batch(s1, s2).tolist() == one.tolist()
    finally:
        api.set_devices(1)


def test_fasta_routes_long_pairs_through_the_long_bucket(monkeypatch):
    r = np.random.default_rng(16)
    s1, s2 = [], []
    for k in range(96):
        if k % 3 == 0:                                           # reads against windows: the batch kernel
            w = rng.random_acgt(16, 2 * k, 800); s1.append(bytes(w[100:250])); s2.append(bytes(w))
        else:                                                    # 2-4 kb records, enough for the multi-band kernel
            a = rng.random_acgt(16, 2 * k, int(r.integers(2000, 4001)))
            b = rng.mutate(a, 16, 2 * k + 1, 0.08, 0.03) if k % 2 else rng.random_acgt(16, 2 * k + 1, int(r.integers(2000, 4001)))
            s1.append(bytes(a)); s2.append(bytes(b))
    ran = []
    orig = api.PackedBatch.score_long
    monkeypatch.setattr(api.PackedBatch, "score_long", lambda self, *a, **k: (ran.append(self.npairs), orig(self, *a, **k))[1])
    got = fasta.score_pairs(s1, s2)
    assert got.tolist() == [api.score(a, b) for a, b in zip(s1, s2)]
    assert ran == [64]
    q = bytes(rng.mutate(rng.random_acgt(17, 0, 3000), 17, 1, 0.05, 0.02))
    db = [bytes(rng.random_acgt(17, 10 + k, 2000 + 30 * k)) for k in range(64)] + [bytes(q[500:2500])]
    ran.clear()
    assert fasta.search(q, db).tolist() == [api.score(q, d) for d in db]
    assert ran == [len(db)]
