"""Batch alignment on the GPU (swb200_align_batch, swb200_batch_align, api.align_batch, fasta.align_pairs): every pair
gets exactly what api.align (swb200_align) returns for it alone."""
import re

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

pytestmark = pytest.mark.gpu

PARAMS = [O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (1, -1, 0, 0), (5, -4, 11, 1)]


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


def _mixed_pairs(seed, n=240):
    """Empty sequences, score-0 pairs, short sides 1 .. 1024, long sides up to 4096, planted and random, both orders."""
    r = np.random.default_rng(seed)
    s1, s2 = [b"", b"ACGT", b"AAAA", b"A" * 1024], [b"ACGT", b"", b"CCCC", b"A" * 4096]
    for k in range(n - len(s1)):
        short = int(r.choice([1, 5, 37, 150, 151, 300, 640, 1024])) if k % 4 else int(r.integers(1, 1025))
        long_ = int(r.integers(short, min(4096, 4 * short + 200) + 1))
        w = rng.random_acgt(seed, 2 * k, long_)
        if k % 2 == 0 and long_ > short > 4:
            o = int(r.integers(0, long_ - short + 1))
            rd = rng.mutate(w[o:o + short], seed, 2 * k + 1, 0.05, 0.02)[:short]     # insertions may lengthen it
        else:
            rd = rng.random_acgt(seed, 2 * k + 1, short)
        a, b = (bytes(rd), bytes(w)) if k % 3 else (bytes(w), bytes(rd))
        s1.append(a); s2.append(b)
    return s1, s2


@pytest.mark.parametrize("p", PARAMS)
def test_align_batch_equals_align(p):
    from concurrentproject_b200 import api
    s1, s2 = _mixed_pairs(500 + PARAMS.index(p))
    scores, spans, cigars = api.align_batch(s1, s2, p)
    for k, (a, b) in enumerate(zip(s1, s2)):
        got = (int(scores[k]), tuple(int(x) for x in spans[k]), cigars[k])
        try:
            want = api.align(a, b, p)
        except api.SwbError as e:
            # gap_ext > gap_init: swb200_align merges two neighbouring opened gaps into one CIGAR run and then refuses it
            # in its own re-score; the batch call reports them as two operations (see include/swb200.h)
            assert p[3] > p[2] and "internal" in str(e)
            assert (got[0],) + got[1] == api.score_span(a, b, p)
            want = got
        assert got == want, (k, p, len(a), len(b), got[0], got[1], want[0], want[1])
        if got[0] > 0:
            aa, bb = np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8)
            assert _rescore(got[2], aa, bb, got[1], p) == (got[0], True)


def test_ops_overflow_and_retry():
    from concurrentproject_b200 import api
    s1, s2 = _mixed_pairs(77, 120)
    p = (2, -3, 5, 1)
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    want = [api.align(a, b, p) for a, b in zip(s1, s2)]
    nops = [len(re.findall(r"\d+[=XID]", w[2])) for w in want]
    scores, spans, ops, cnt = api.align_batch_ops(f1, o1, l1, f2, o2, l2, p, ops_stride=3)
    assert any(n > 3 for n in nops) and any(0 < n <= 3 for n in nops)
    for k, w in enumerate(want):
        assert (int(scores[k]), tuple(int(x) for x in spans[k])) == w[:2]
        if nops[k] > 3:
            assert cnt[k] == -nops[k] and not ops[k].any()           # overflow: reported, nothing written
        else:
            assert cnt[k] == nops[k] and api.cigar_string(ops[k, :cnt[k]]) == w[2]
    # the Python wrapper redoes the overflowed pairs with room for len1 + len2 operations
    sc2, sp2, cig2 = api.align_batch(s1, s2, p, ops_stride=3)
    assert [(int(sc2[k]), tuple(int(x) for x in sp2[k]), cig2[k]) for k in range(len(s1))] == want


def test_errors_match_score_batch():
    from concurrentproject_b200 import api
    good1, good2 = [b"ACGT" * 10, b"ACG"], [b"ACGA" * 12, b"TTACG"]
    cases = [
        (good1 + [b"ACNGT"], good2 + [b"ACGT"], O.DEFAULT),           # alphabet
        (good1 + [b"A" * 1100], good2 + [b"C" * 1100], O.DEFAULT),    # short side over 1024
        (good1 + [b"A" * 800], good2 + [b"A" * 900], (50, -1, 1, 1)),  # match * min(len) out of range
        (good1, good2, (1, 1, 1, 1)),                                 # parameters
    ]
    for s1, s2, p in cases:
        with pytest.raises(api.SwbError) as e1:
            api.score_batch(s1, s2, p)
        with pytest.raises(api.SwbError) as e2:
            api.align_batch(s1, s2, p)
        assert e1.value.code == e2.value.code, (e1.value, e2.value)


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


def test_cfg4_sample():
    """100 000 read pairs of BASELINE config 4: scores equal swb200_batch_score's, 500 sampled pairs equal api.align,
    and the device-resident call equals the host call."""
    import torch
    from concurrentproject_b200 import api
    n = 100_000
    reads, wins, o1, o2, l1, l2 = _cfg4(torch, n)
    ctx = api.Context(0)
    try:
        pb = api.PackedBatch(ctx, reads.data_ptr(), o1.data_ptr(), l1.data_ptr(), wins.data_ptr(), o2.data_ptr(), l2.data_ptr(), n,
                             150, 1000, n * 150 * 1000)
        d_ref = torch.empty(n, dtype=torch.int32, device="cuda")
        d_sc = torch.empty(n, dtype=torch.int32, device="cuda")
        d_sp = torch.empty((n, 4), dtype=torch.int32, device="cuda")
        d_ops = torch.empty((n, 1150), dtype=torch.int32, device="cuda")
        d_cnt = torch.empty(n, dtype=torch.int32, device="cuda")
        pb.score(d_ref.data_ptr())
        pb.align(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), 1150, d_cnt.data_ptr())
        info = api.last_run(ctx)
        pb.close()
    finally:
        ctx.close()
    assert torch.equal(d_sc, d_ref)
    assert info["engine_launches"] >= 2 and info["cells"] >= n * 150 * 1000
    sc, sp, ops, cnt = d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_ops.cpu().numpy().view(np.uint32), d_cnt.cpu().numpy()
    assert (cnt >= 0).all()
    hr, hw = reads.cpu().numpy(), wins.cpu().numpy()
    for k in np.random.default_rng(1).choice(n, 500, replace=False).tolist():
        a, b = hr[k * 150:(k + 1) * 150], hw[k * 1000:(k + 1) * 1000]
        assert (int(sc[k]), tuple(int(x) for x in sp[k]), api.cigar_string(ops[k, :cnt[k]])) == api.align(a, b), k
    # host call: copy, pack and align in chunks
    ho1, ho2 = np.arange(n, dtype=np.int64) * 150, np.arange(n, dtype=np.int64) * 1000
    hl1, hl2 = np.full(n, 150, np.int32), np.full(n, 1000, np.int32)
    sc2, sp2, ops2, cnt2 = api.align_batch_ops(hr, ho1, hl1, hw, ho2, hl2, api.DEFAULT_PARAMS, ops_stride=1150)
    assert np.array_equal(sc2, sc) and np.array_equal(sp2, sp) and np.array_equal(cnt2, cnt)
    mask = np.arange(1150)[None, :] < cnt[:, None]
    assert np.array_equal(ops2[mask], ops[mask])


def test_two_gpus_identical():
    import torch
    from concurrentproject_b200 import api
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _mixed_pairs(900, 300)
    p = (2, -3, 5, 1)
    one = api.align_batch(s1, s2, p)
    api.set_devices(2)
    try:
        two = api.align_batch(s1, s2, p)
    finally:
        api.set_devices(1)
    assert np.array_equal(one[0], two[0]) and np.array_equal(one[1], two[1]) and one[2] == two[2]


def test_fasta_align_pairs():
    """Batchable pairs, pairs with N, pairs with a short side over 1024: each equals api.align."""
    from concurrentproject_b200 import api, fasta
    s1, s2 = _mixed_pairs(31, 60)
    s1 += [b"ACGTNACGTACGT", bytes(rng.random_acgt(8, 0, 1200)), b"NNNN", b""]
    x = rng.random_acgt(8, 0, 1500)
    s2 += [b"ACGTACGTACGT", bytes(rng.mutate(x, 8, 1, 0.05, 0.02)[:1300]), b"", b"ACGN"]
    scores, spans, cigars = fasta.align_pairs(s1, s2, O.DEFAULT, min_bucket=8)
    for k, (a, b) in enumerate(zip(s1, s2)):
        assert (int(scores[k]), tuple(int(v) for v in spans[k]), cigars[k]) == api.align(a, b), k
