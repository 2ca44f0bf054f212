"""Banded batch alignment on the GPU (swb200_align_banded_batch, swb200_batch_align_banded, api.align_banded_batch,
PackedBatch.align_banded): scores equal the banded score-only call, spans equal the C checker (banded_oracle), and every
CIGAR re-scores to the score, consumes exactly the span and stays inside the band."""
import re

import numpy as np
import pytest

import banded_oracle as BO
import oracle_lib as O
from concurrentproject_b200 import rng

pytestmark = pytest.mark.gpu

PARAMS = [O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (1, -1, 0, 0), (5, -4, 11, 1)]
_OPC = {"=": 0, "X": 1, "I": 2, "D": 3}


def check_cigar(cigar, a, b, span, p, lo, hi):
    """(re-score, consumes exactly the span, every visited cell in lo <= j - i <= hi), vectorised for 10 kb pairs."""
    ma, mi, gi, ge = p
    runs = [(int(c), op) for c, op in re.findall(r"(\d+)([=XID])", cigar)]
    cnt = np.array([c for c, _ in runs], np.int64)
    code = np.array([_OPC[op] for _, op in runs], np.int64)
    per = np.repeat(code, cnt)                                  # one entry per visited cell
    di = np.where((per == 0) | (per == 1) | (per == 3), 1, 0)
    dj = np.where((per == 0) | (per == 1) | (per == 2), 1, 0)
    i = span[0] + np.concatenate([[0], np.cumsum(di)[:-1]])     # 1-based cell of each operation character
    j = span[1] + np.concatenate([[0], np.cumsum(dj)[:-1]])
    diag = per <= 1
    eq = a[j[diag] - 1] == b[i[diag] - 1]
    pairs_ok = bool(np.array_equal(eq, per[diag] == 0))
    total = int(ma * (per == 0).sum() + mi * (per == 1).sum() - (gi * ((code >= 2).sum()) + ge * (cnt[code >= 2] - 1).sum()))
    ends = (int(i[-1]), int(j[-1])) == (span[2], span[3]) if len(per) else False
    in_band = bool(((j - i >= lo) & (j - i <= hi)).all())
    return (total if pairs_ok else None), ends, in_band


def _check(s1, s2, scores, spans, cigars, lo, hi, p):
    from concurrentproject_b200 import api
    assert np.array_equal(scores, api.score_banded_batch(s1, s2, lo, hi, p))
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = BO.gotoh_banded_span(a, b, lo, hi, p)
        assert (int(scores[k]),) + tuple(int(x) for x in spans[k]) == want, (k, lo, p)
        if want[0] > 0:
            aa, bb = np.frombuffer(bytes(a), np.uint8), np.frombuffer(bytes(b), np.uint8)
            assert check_cigar(cigars[k], aa, bb, spans[k], p, lo, hi) == (want[0], True, True), (k, lo, p)
        else:
            assert cigars[k] == ""


def _mixed_pairs(seed, n):
    """Empty sequences, pairs shorter than the band, reads against windows, long related pairs with a drift, random."""
    r = np.random.default_rng(seed)
    s1, s2 = [b"", b"ACGT", b"A" * 30], [b"ACGT", b"", b"A" * 25]
    for k in range(n - len(s1)):
        m = int(r.choice([8, 40, 150, 600, 2000, 5000])) if k % 3 else int(r.integers(1, 3000))
        src = rng.random_acgt(seed, 2 * k, m + 200)
        if k % 5 == 4:
            a, b = src[:m], rng.random_acgt(seed, 2 * k + 1, int(r.integers(1, m + 1)))
        else:
            sh = int(r.integers(-40, 41))
            b = rng.mutate(src, seed, 2 * k + 1, 0.08, 0.03)
            a, b = (src[sh:sh + m], b[:m]) if sh >= 0 else (src[:m], b[-sh:m - sh])
        s1.append(bytes(a)); s2.append(bytes(b))
    return s1, s2


@pytest.mark.parametrize("p", PARAMS)
def test_mixed_pairs_each_parameter_set(p):
    from concurrentproject_b200 import api
    s1, s2 = _mixed_pairs(600 + PARAMS.index(p), 50)
    for lo in (-32, -10, -53, 7):
        scores, spans, cigars = api.align_banded_batch(s1, s2, lo, lo + 63, p)
        _check(s1, s2, scores, spans, cigars, lo, lo + 63, p)


@pytest.mark.parametrize("p", PARAMS)
def test_full_band_equals_align_batch(p):
    """Pairs that fit inside the band: the result is align_batch's."""
    from concurrentproject_b200 import api
    r = np.random.default_rng(700 + PARAMS.index(p))
    s1, s2 = [], []
    for k in range(80):
        n, m = int(r.integers(0, 33)), int(r.integers(0, 32))
        a = rng.random_acgt(70, 2 * k, n)
        b = rng.mutate(a, 70, 2 * k + 1, 0.1, 0.05)[:m] if k % 2 else rng.random_acgt(70, 2 * k + 1, m)
        s1.append(bytes(a)); s2.append(bytes(b))
    for lo in (-31, -32):
        got = api.align_banded_batch(s1, s2, lo, lo + 63, p)
        want = api.align_batch(s1, s2, p)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]


def _cfg5(torch, npairs, length=10000, seed=5):
    from concurrentproject_b200 import api
    dev = torch.device("cuda", 0)
    d1 = torch.empty(npairs * length, dtype=torch.uint8, device=dev)
    d2 = torch.empty(npairs * length, dtype=torch.uint8, device=dev)
    api.gen_long_pairs_device(0, seed, 0, npairs, length, d1.data_ptr(), d2.data_ptr())
    torch.cuda.synchronize()
    off = torch.arange(npairs, dtype=torch.int64, device=dev) * length
    ln = torch.full((npairs,), length, dtype=torch.int32, device=dev)
    return d1, d2, off, ln


def test_cfg5_pairs_host_and_device():
    """2 000 cfg5 pairs (10 kb, band -32..31): the device-resident call equals the host call word for word, scores equal
    the banded score-only call, and every pair's span and CIGAR check out against the C checker."""
    import torch
    from concurrentproject_b200 import api
    n, L, lo, hi, stride = 2000, 10000, -32, 31, 8192
    d1, d2, off, ln = _cfg5(torch, n, L)
    ctx = api.Context(0)
    try:
        pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n,
                             L, L, n * L * 64, keep_order=True)
        d_ref = torch.empty(n, dtype=torch.int32, device="cuda")
        d_sc = torch.empty(n, dtype=torch.int32, device="cuda")
        d_sp = torch.empty((n, 4), dtype=torch.int32, device="cuda")
        d_ops = torch.zeros((n, stride), dtype=torch.int32, device="cuda")
        d_cnt = torch.empty(n, dtype=torch.int32, device="cuda")
        pb.score_banded(d_ref.data_ptr(), lo, hi)
        pb.align_banded(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), stride, d_cnt.data_ptr(), lo, hi)
        info = api.last_run(ctx)
        pb.close()
    finally:
        ctx.close()
    assert torch.equal(d_sc, d_ref)
    assert info["config"] == 310 and info["engine_launches"] >= 2 and info["cells"] >= n * L * 60
    sc, sp, ops, cnt = d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_ops.cpu().numpy().view(np.uint32), d_cnt.cpu().numpy()
    assert (cnt > 0).all()
    h1, h2 = d1.cpu().numpy(), d2.cpu().numpy()
    ho, hl = np.arange(n, dtype=np.int64) * L, np.full(n, L, np.int32)
    sc2, sp2, ops2, cnt2 = api.align_banded_batch_ops(h1, ho, hl, h2, ho.copy(), hl.copy(), lo, hi, api.DEFAULT_PARAMS, stride)
    assert np.array_equal(sc2, sc) and np.array_equal(sp2, sp) and np.array_equal(cnt2, cnt) and np.array_equal(ops2, ops)
    for k in range(n):
        a, b = h1[k * L:(k + 1) * L], h2[k * L:(k + 1) * L]
        want = BO.gotoh_banded_span(a, b, lo, hi)
        assert (int(sc[k]),) + tuple(int(x) for x in sp[k]) == want, k
        assert check_cigar(api.cigar_string(ops[k, :cnt[k]]), a, b, sp[k], api.DEFAULT_PARAMS, lo, hi) == (want[0], True, True), k


def test_ops_overflow_and_retry():
    from concurrentproject_b200 import api
    s1, s2 = _mixed_pairs(77, 60)
    p, lo, hi = (2, -3, 5, 1), -32, 31
    full = api.align_banded_batch(s1, s2, lo, hi, p, ops_stride=20000)
    nops = [len(re.findall(r"\d+[=XID]", c)) for c in full[2]]
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    scores, spans, ops, cnt = api.align_banded_batch_ops(f1, o1, l1, f2, o2, l2, lo, hi, p, ops_stride=5)
    assert any(x > 5 for x in nops) and any(0 < x <= 5 for x in nops)
    assert np.array_equal(scores, full[0]) and np.array_equal(spans, full[1])
    for k, x in enumerate(nops):
        if x > 5:
            assert cnt[k] == -x and not ops[k].any()                  # overflow: reported, slot zero-filled
        else:
            assert cnt[k] == x and api.cigar_string(ops[k, :cnt[k]]) == full[2][k]
    again = api.align_banded_batch(s1, s2, lo, hi, p, ops_stride=5)   # the wrapper redoes the overflowed pairs
    assert np.array_equal(again[0], full[0]) and np.array_equal(again[1], full[1]) and again[2] == full[2]


def test_errors_match_score_banded_batch():
    from concurrentproject_b200 import api
    good1, good2 = [b"ACGT" * 10, b"ACG"], [b"ACGA" * 12, b"TTACG"]
    cases = [
        (good1 + [b"ACNGT"], good2 + [b"ACGT"], -32, 31, O.DEFAULT),          # alphabet
        (good1, good2, -32, 40, O.DEFAULT),                                  # band width
        (good1 + [b"A" * 800], good2 + [b"A" * 900], -32, 31, (50, -1, 1, 1)),  # match * min(len) out of range
        (good1, good2, -32, 31, (1, 1, 1, 1)),                               # parameters
    ]
    for s1, s2, lo, hi, p in cases:
        with pytest.raises(api.SwbError) as e1:
            api.score_banded_batch(s1, s2, lo, hi, p)
        with pytest.raises(api.SwbError) as e2:
            api.align_banded_batch(s1, s2, lo, hi, p)
        assert e1.value.code == e2.value.code, (e1.value, e2.value)
    with pytest.raises(api.SwbError) as e:
        api.align_banded_batch(good1 + [b"ACNGT"], good2 + [b"ACGT"])
    assert e.value.code == -3


def test_device_call_refuses_a_read_batch_layout():
    import torch
    from concurrentproject_b200 import api
    d1, d2, off, ln = _cfg5(torch, 4, 200)
    ctx = api.Context(0)
    try:
        pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), 4,
                             200, 200, 4 * 200 * 200, keep_order=False)
        out = torch.zeros(64, dtype=torch.int32, device="cuda")
        with pytest.raises(api.SwbError) as e:
            pb.align_banded(out.data_ptr(), out.data_ptr(), out.data_ptr(), 4, out.data_ptr())
        assert e.value.code == -2
        pb.close()
    finally:
        ctx.close()


def test_two_gpus_identical():
    import torch
    from concurrentproject_b200 import api
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _mixed_pairs(900, 120)
    p = (2, -3, 5, 1)
    one = api.align_banded_batch(s1, s2, -32, 31, p)
    api.set_devices(2)
    try:
        two = api.align_banded_batch(s1, s2, -32, 31, p)
    finally:
        api.set_devices(1)
    assert np.array_equal(one[0], two[0]) and np.array_equal(one[1], two[1]) and one[2] == two[2]
