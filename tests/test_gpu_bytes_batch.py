"""Byte batches on the GPU (swb200_score_batch_bytes, swb200_align_batch_bytes, swb200_batch_pack_device_bytes, and the
fasta routes that use them): every pair gets what the single-pair calls give it alone, on any bytes; on A,C,G,T the byte
calls equal the 2-bit batch calls exactly; every form of the call (host, device, chunked, shuffled offsets, a shared
seq1 buffer, two GPUs) gives the same result."""
import re

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

pytestmark = pytest.mark.gpu

ALPHABETS = [b"ACGTN", b"ACGTRYSWKMBDHVN", b"ACDEFGHIKLMNPQRSTVWY", bytes(range(256))]


def _rescore(cigar, a, b, span, p):
    ma, mi, gi, ge = p
    i, j, total = span[0] - 1, span[1] - 1, 0
    for cnt, op in re.findall(r"(\d+)([=XID])", cigar):
        cnt = int(cnt)
        if op in "=X":
            assert all((a[j + t] == b[i + t]) == (op == "=") for t in range(cnt))
            total += cnt * (ma if op == "=" else mi)
            i, j = i + cnt, j + cnt
        else:
            total -= gi + (cnt - 1) * ge
            if op == "I":
                j += cnt
            else:
                i += cnt
    return total, (i, j) == (span[2], span[3])


def _ragged(seed, n):
    """n ragged pairs, a quarter from each alphabet: short sides 0 .. 1024, long sides up to 2048, half planted with
    substitutions from the alphabet, both orders; empty sequences and score-0 pairs among them."""
    r = np.random.default_rng(seed)
    s1, s2 = [b"", b"NNNN", b"\x00\x04\xff", b"n" * 10], [b"ACGN", b"", b"\x04\x00", b"N" * 10]
    for k in range(n - len(s1)):
        alpha = np.frombuffer(ALPHABETS[k % 4], np.uint8)
        short = int(r.choice([1, 7, 64, 150, 300, 1024])) if k % 3 else int(r.integers(1, 1025))
        long_ = int(r.integers(short, min(2048, 3 * short + 100) + 1))
        w = alpha[r.integers(0, len(alpha), long_)]
        if k % 2 == 0 and long_ > short > 4:
            o = int(r.integers(0, long_ - short + 1))
            rd = w[o:o + short].copy()
            sub = r.random(short) < 0.06
            rd[sub] = alpha[r.integers(0, len(alpha), int(sub.sum()))]
        else:
            rd = alpha[r.integers(0, len(alpha), short)]
        a, b = (rd.tobytes(), w.tobytes()) if k % 3 else (w.tobytes(), rd.tobytes())
        s1.append(a); s2.append(b)
    return s1, s2


def _check_align(got, a, b, p):
    try:
        want = _align(a, b, p)
    except Exception as e:
        # gap_ext > gap_init: swb200_align merges two neighbouring opened gaps into one CIGAR run and then refuses it in
        # its own re-score; the batch call reports them as two operations (include/swb200.h)
        from concurrentproject_b200 import api
        assert p[3] > p[2] and "internal" in str(e)
        assert (got[0],) + got[1] == api.score_span(a, b, p)
        want = got
    assert got == want, (len(a), len(b), got[0], got[1], want[0], want[1])
    if got[0] > 0:
        assert _rescore(got[2], np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8), got[1], p) == (got[0], True)


def _align(a, b, p):
    from concurrentproject_b200 import api
    return api.align(a, b, p)


@pytest.mark.parametrize("p", [O.DEFAULT, (2, -1, 1, 3), (5, -4, 11, 1)])
def test_ragged_any_bytes(p):
    """3 000 ragged pairs with N, IUPAC, protein and all-byte content: every score equals the oracle's; 200 sampled pairs
    (and the special ones) equal api.align in score, span and CIGAR."""
    from concurrentproject_b200 import api
    s1, s2 = _ragged(700 + p[0], 3000)
    want = O.gotoh_batch(s1, s2, p)
    assert np.array_equal(api.score_batch_bytes(s1, s2, p), want)
    assert api.last_run()["config"] == 101
    scores, spans, cigars = api.align_batch_bytes(s1, s2, p)
    assert api.last_run()["config"] == 301
    assert np.array_equal(scores, want)
    for k in list(range(4)) + np.random.default_rng(p[0]).choice(len(s1), 200, replace=False).tolist():
        _check_align((int(scores[k]), tuple(int(x) for x in spans[k]), cigars[k]), s1[k], s2[k], p)


def _cfg4(torch, npairs, seed=4):
    from concurrentproject_b200 import api
    dev = torch.device("cuda", 0)
    reads = torch.empty(npairs * 150, dtype=torch.uint8, device=dev)
    wins = torch.empty(npairs * 1000, dtype=torch.uint8, device=dev)
    api.gen_read_pairs_device(0, seed, 0, npairs, 150, 1000, reads.data_ptr(), wins.data_ptr())
    torch.cuda.synchronize()
    o1 = torch.arange(npairs, dtype=torch.int64, device=dev) * 150
    o2 = torch.arange(npairs, dtype=torch.int64, device=dev) * 1000
    l1 = torch.full((npairs,), 150, dtype=torch.int32, device=dev)
    l2 = torch.full((npairs,), 1000, dtype=torch.int32, device=dev)
    return reads, wins, o1, o2, l1, l2


def test_cfg4_acgt_equals_two_bit_and_other_calls_refuse():
    """100 000 cfg4 pairs (A,C,G,T only): the byte batch's scores, spans and operations equal the 2-bit batch's exactly,
    device-resident and from host buffers; the four calls without a byte kernel refuse the byte batch."""
    import torch
    from concurrentproject_b200 import api
    n, stride = 100_000, 1150
    reads, wins, o1, o2, l1, l2 = _cfg4(torch, n)
    ctx = api.Context(0)
    out = {}
    try:
        for by in (False, True):
            pb = api.PackedBatch(ctx, reads.data_ptr(), o1.data_ptr(), l1.data_ptr(), wins.data_ptr(), o2.data_ptr(), l2.data_ptr(),
                                 n, 150, 1000, n * 150 * 1000, byte_symbols=by)
            try:
                d = [torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda"),
                     torch.zeros((n, 4), dtype=torch.int32, device="cuda"), torch.zeros((n, stride), dtype=torch.int32, device="cuda"),
                     torch.zeros(n, dtype=torch.int32, device="cuda")]
                pb.score(d[0].data_ptr())
                assert (api.last_run(ctx)["config"] == 101) == by
                pb.align(d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), stride, d[4].data_ptr())
                assert api.last_run(ctx)["config"] == (301 if by else 300)
                out[by] = [x.cpu().numpy() for x in d]
                if by:
                    p = api.DEFAULT_PARAMS
                    for call in (lambda: pb.score_long(d[0].data_ptr(), p), lambda: pb.score_banded(d[0].data_ptr(), -32, 31, p),
                                 lambda: pb.align_banded(d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), stride, d[4].data_ptr()),
                                 lambda: pb.align_long(d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), stride, d[4].data_ptr())):
                        with pytest.raises(api.SwbError) as e:
                            call()
                        assert e.value.code == -2 and "bytes" in str(e.value)
            finally:
                pb.close()
    finally:
        ctx.close()
    for a, b in zip(out[False], out[True]):
        assert np.array_equal(a, b)
    sc, sp, ops, cnt = out[True][1], out[True][2], out[True][3].view(np.uint32), out[True][4]
    assert np.array_equal(out[True][0], sc) and (cnt >= 0).all()
    # the host calls: copy, pack and run in chunks
    hr, hw = reads.cpu().numpy(), wins.cpu().numpy()
    ho1, ho2 = np.arange(n, dtype=np.int64) * 150, np.arange(n, dtype=np.int64) * 1000
    hl1, hl2 = np.full(n, 150, np.int32), np.full(n, 1000, np.int32)
    assert np.array_equal(api.score_batch_bytes_flat(hr, ho1, hl1, hw, ho2, hl2), sc)
    sc2, sp2, ops2, cnt2 = api.align_batch_bytes_ops(hr, ho1, hl1, hw, ho2, hl2, api.DEFAULT_PARAMS, ops_stride=stride)
    assert np.array_equal(sc2, sc) and np.array_equal(sp2, sp) and np.array_equal(cnt2, cnt)
    mask = np.arange(stride)[None, :] < cnt[:, None]
    assert np.array_equal(ops2[mask], ops[mask])


def test_forms_agree():
    """Host call = device call; forced small chunks, offsets out of order and one shared seq1 buffer change nothing."""
    import torch
    from concurrentproject_b200 import api
    p = (2, -3, 5, 1)
    s1, s2 = _ragged(41, 900)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    want_sc = api.score_batch_bytes_flat(f1, o1, l1, f2, o2, l2, p)
    want = api.align_batch_bytes_ops(f1, o1, l1, f2, o2, l2, p, 2048)
    assert np.array_equal(want_sc, want[0]) and np.array_equal(want_sc, O.gotoh_batch(s1, s2, p))
    api.configure("batch_chunk_bytes", "20000")
    try:
        assert np.array_equal(api.score_batch_bytes_flat(f1, o1, l1, f2, o2, l2, p), want_sc)
        assert all(np.array_equal(a, b) for a, b in zip(api.align_batch_bytes_ops(f1, o1, l1, f2, o2, l2, p, 2048), want))
    finally:
        api.configure("batch_chunk_bytes", "0")
    # offsets out of order: the same pairs laid out in reverse in the flat buffers
    rev1, ro1, rl1 = api._flatten(s1[::-1])
    rev2, ro2, rl2 = api._flatten(s2[::-1])
    ro1, ro2 = ro1[::-1].copy(), ro2[::-1].copy()
    assert np.array_equal(api.score_batch_bytes_flat(rev1, ro1, l1, rev2, ro2, l2, p), want_sc)
    assert all(np.array_equal(a, b) for a, b in zip(api.align_batch_bytes_ops(rev1, ro1, l1, rev2, ro2, l2, p, 2048), want))
    # one shared seq1 buffer: every pair's seq1 and seq2 cut from the same bytes
    allb = np.concatenate([f1, f2])
    o2s = o2 + len(f1)
    assert np.array_equal(api.score_batch_bytes_flat(allb, o1, l1, allb, o2s, l2, p), want_sc)
    # device-resident batch over the same buffer
    ctx = api.Context(0)
    try:
        d_all = torch.from_numpy(allb).cuda()
        d = [torch.from_numpy(x).cuda() for x in (o1, l1, o2s, l2)]
        n = len(l1)
        pb = api.PackedBatch(ctx, d_all.data_ptr(), d[0].data_ptr(), d[1].data_ptr(), d_all.data_ptr(), d[2].data_ptr(),
                             d[3].data_ptr(), n, int(np.minimum(l1, l2).max()), int(np.maximum(l1, l2).max()), 0,
                             byte_symbols=True)
        try:
            d_sc = torch.zeros(n, dtype=torch.int32, device="cuda")
            d_sp = torch.zeros((n, 4), dtype=torch.int32, device="cuda")
            d_ops = torch.zeros((n, 2048), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
            pb.score(d_sc.data_ptr(), p)
            assert np.array_equal(d_sc.cpu().numpy(), want_sc)
            pb.align(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), 2048, d_cnt.data_ptr(), p)
        finally:
            pb.close()
    finally:
        ctx.close()
    assert np.array_equal(d_sc.cpu().numpy(), want[0]) and np.array_equal(d_sp.cpu().numpy(), want[1])
    assert np.array_equal(d_cnt.cpu().numpy(), want[3]) and np.array_equal(d_ops.cpu().numpy().view(np.uint32), want[2])
    with pytest.raises(ValueError):
        api.PackedBatch(None, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, keep_order=True, byte_symbols=True)


def test_two_gpus_identical():
    import torch
    from concurrentproject_b200 import api
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _ragged(900, 600)
    p = (2, -3, 5, 1)
    one = (api.score_batch_bytes(s1, s2, p), api.align_batch_bytes(s1, s2, p))
    api.set_devices(2)
    try:
        two = (api.score_batch_bytes(s1, s2, p), api.align_batch_bytes(s1, s2, p))
    finally:
        api.set_devices(1)
    assert np.array_equal(one[0], two[0])
    assert np.array_equal(one[1][0], two[1][0]) and np.array_equal(one[1][1], two[1][1]) and one[1][2] == two[1][2]


def test_fasta_routes_bytes_through_the_byte_batch(monkeypatch):
    """score_pairs, search and align_pairs on inputs with N, IUPAC and lower-case bytes equal the oracle / api.align, and
    no such pair goes through the per-pair calls: they run on byte batches."""
    from concurrentproject_b200 import api, fasta
    s1, s2 = _ragged(55, 120)
    x = rng.random_acgt(8, 0, 1500)
    s1 += [b"ACGTNACGTACGT", bytes(x[:1200]) + b"N", b"acgt"]         # the long pair with an N stays on the single-pair engine
    s2 += [b"ACGTACGTACGT", bytes(rng.mutate(x, 8, 1, 0.05, 0.02)[:1300]), b"ACGT"]
    calls, packs = {"score": 0, "align": 0}, []
    real_score, real_align, real_init = api.Context.score_device, api.Context.align_device, api.PackedBatch.__init__

    def count_score(self, *a, **k):
        calls["score"] += 1
        return real_score(self, *a, **k)

    def count_align(self, *a, **k):
        calls["align"] += 1
        return real_align(self, *a, **k)

    def record(self, *a, byte_symbols=False, **k):
        packs.append((a[7], byte_symbols))
        return real_init(self, *a, byte_symbols=byte_symbols, **k)

    monkeypatch.setattr(api.Context, "score_device", count_score)
    monkeypatch.setattr(api.Context, "align_device", count_align)
    monkeypatch.setattr(api.PackedBatch, "__init__", record)
    p = O.DEFAULT
    assert np.array_equal(fasta.score_pairs(s1, s2, p, min_bucket=8), O.gotoh_batch(s1, s2, p))
    assert calls["score"] == 1                                          # the one long pair with an N
    assert any(by for _, by in packs)
    query = b"ACGTNNACGTRYACGTAAAACCCCGGGGTTTTN"
    db = [w for w in s2 if len(w) <= 1024]
    calls["score"] = 0
    assert np.array_equal(fasta.search(query, db, p, min_bucket=8), O.gotoh_batch([query] * len(db), db, p))
    assert calls["score"] == 0
    packs.clear()
    scores, spans, cigars = fasta.align_pairs(s1, s2, p, min_bucket=8)
    assert calls["align"] == 1 and any(by for _, by in packs)
    for k, (a, b) in enumerate(zip(s1, s2)):
        assert (int(scores[k]), tuple(int(v) for v in spans[k]), cigars[k]) == api.align(a, b, p), k
