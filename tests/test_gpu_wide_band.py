"""Bands of 128, 256 and 512 diagonals on the GPU through the C ABI: scores of every banded call (host, host-packed,
device batch, single pair) equal oracle_gotoh_banded_batch; alignments have the C checker's score and span and CIGARs
that re-score to the score inside the band; the ops_stride overflow path; refusals of other widths; run info."""
import ctypes as C

import numpy as np
import pytest

import banded_oracle as BO
import oracle_lib as O
from concurrentproject_b200 import rng
from test_gpu_align_banded import _check, _mixed_pairs, check_cigar

pytestmark = pytest.mark.gpu

WIDTHS = [128, 256, 512]
PARAMS = [O.DEFAULT, (2, -3, 5, 1), (2, -1, 1, 3)]


def _drift_pairs(seed, n, W):
    """_mixed_pairs plus related pairs whose best alignment drifts by up to W/2 diagonals (planted deletions)."""
    s1, s2 = _mixed_pairs(seed, n)
    r = np.random.default_rng(seed)
    for k in range(12):
        m, cut = int(r.integers(400, 3000)), int(r.integers(10, W // 2))
        a = rng.random_acgt(seed + 1, k, m)
        b = rng.mutate(np.concatenate([a[:m // 2], a[m // 2 + cut:]]), seed + 1, 100 + k, 0.05, 0.02)
        s1.append(bytes(a)); s2.append(bytes(b))
    return s1, s2


def _single(a, b, lo, hi, p):
    from concurrentproject_b200 import _lib
    out = C.c_int(-1)
    pp = _lib.Params(*p)
    buf1, buf2 = (C.c_ubyte * max(1, len(a))).from_buffer_copy(a or b"A"), (C.c_ubyte * max(1, len(b))).from_buffer_copy(b or b"A")
    rc = _lib.load().swb200_score_banded(buf1, len(a), buf2, len(b), lo, hi, C.byref(pp), C.byref(out))
    return rc, out.value


def _packed(s1, s2, lo, hi, p):
    """swb200_score_banded_batch_packed on the host-packed batch."""
    from concurrentproject_b200 import api
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    w1, st1, w2, st2 = api.pack_banded_host(f1, o1, l1, f2, o2, l2)
    return api.score_banded_batch_packed(w1, st1, w2, st2, l1, l2, lo, hi, p)


def _device_scores(torch, s1, s2, lo, hi, p):
    from concurrentproject_b200 import api
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (f1, o1, l1, f2, o2, l2)]
    n = len(s1)
    ctx = api.Context(0)
    try:
        pb = api.PackedBatch(ctx, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                             t[5].data_ptr(), n, int(l1.max()), int(l2.max()), int((l1.astype(np.int64) * l2).sum()),
                             keep_order=True)
        d = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        pb.score_banded(d.data_ptr(), lo, hi, p)
        torch.cuda.synchronize()
        info = api.last_run(ctx)
        pb.close()
    finally:
        ctx.close()
    return d.cpu().numpy(), info


@pytest.mark.parametrize("W", WIDTHS)
def test_scores_through_every_call(W):
    import torch
    from concurrentproject_b200 import api
    s1, s2 = _drift_pairs(1000 + W, 45, W)
    for p in PARAMS:
        for lo in (-W // 2, -W // 2 + 5, -W + 9, 3):
            hi = lo + W - 1
            want = O.gotoh_banded_batch(s1, s2, lo, hi, p)
            assert np.array_equal(api.score_banded_batch(s1, s2, lo, hi, p), want), (W, p, lo)
            info = api.last_run()
            assert info["bands"] == W and info["config"] == 2000 + W
            assert np.array_equal(_packed(s1, s2, lo, hi, p), want), (W, p, lo)
            got, info = _device_scores(torch, s1, s2, lo, hi, p)
            assert np.array_equal(got, want) and info["bands"] == W, (W, p, lo)
    for k in (3, 20, 50):
        assert _single(s1[k], s2[k], -W // 2, W // 2 - 1, (2, -3, 5, 1)) == (0, O.gotoh_banded(s1[k], s2[k], -W // 2, W // 2 - 1, (2, -3, 5, 1)))


def test_many_small_chunks():
    from concurrentproject_b200 import api
    s1, s2 = _drift_pairs(1100, 60, 256)
    want = {W: O.gotoh_banded_batch(s1, s2, -W // 2, W // 2 - 1) for W in WIDTHS}
    api.configure("batch_chunk_bytes", "20000")
    try:
        for W in WIDTHS:
            assert np.array_equal(api.score_banded_batch(s1, s2, -W // 2, W // 2 - 1), want[W]), W
            assert np.array_equal(_packed(s1, s2, -W // 2, W // 2 - 1, O.DEFAULT), want[W]), W
    finally:
        api.configure("batch_chunk_bytes", "0")


@pytest.mark.parametrize("W", WIDTHS)
def test_alignments(W):
    from concurrentproject_b200 import api
    s1, s2 = _drift_pairs(1200 + W, 40, W)
    for p in PARAMS:
        for lo in (-W // 2, -W // 2 + 3):
            scores, spans, cigars = api.align_banded_batch(s1, s2, lo, lo + W - 1, p)
            assert api.last_run()["bands"] == W
            _check(s1, s2, scores, spans, cigars, lo, lo + W - 1, p)


def test_wider_band_recovers_planted_indels():
    """An 80-100 base deletion: W = 64 scores below the unbanded score, W = 256 equals it, score and alignment."""
    from concurrentproject_b200 import api
    s1, s2 = [], []
    for k, cut in enumerate((80, 90, 100)):
        a = rng.random_acgt(1300, k, 3000)
        b = rng.mutate(np.concatenate([a[:1500], a[1500 + cut:]]), 1300, 10 + k, 0.02, 0.0)
        s1.append(bytes(a)); s2.append(bytes(b))
    full = [O.gotoh_full(a, b) for a, b in zip(s1, s2)]
    assert (api.score_banded_batch(s1, s2, -32, 31) < full).all()
    assert api.score_banded_batch(s1, s2, -128, 127).tolist() == full
    assert api.align_banded_batch(s1, s2, -128, 127)[0].tolist() == full


def test_cfg5_device_equals_host():
    """1 000 cfg5 pairs (10 kb) in a 256-diagonal band: the device-resident alignment equals the host call word for word,
    its scores equal the device score call, and sampled pairs check out against the C checker."""
    import torch
    from concurrentproject_b200 import api
    from test_gpu_align_banded import _cfg5
    n, L, lo, hi, stride = 1000, 10000, -128, 127, 8192
    d1, d2, off, ln = _cfg5(torch, n, L)
    ctx = api.Context(0)
    try:
        pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n,
                             L, L, n * L * 256, keep_order=True)
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
    assert info["config"] == 312 and info["bands"] == 256
    sc, sp, ops, cnt = d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_ops.cpu().numpy().view(np.uint32), d_cnt.cpu().numpy()
    assert (cnt > 0).all()
    h1, h2 = d1.cpu().numpy(), d2.cpu().numpy()
    ho, hl = np.arange(n, dtype=np.int64) * L, np.full(n, L, np.int32)
    sc2, sp2, ops2, cnt2 = api.align_banded_batch_ops(h1, ho, hl, h2, ho.copy(), hl.copy(), lo, hi, api.DEFAULT_PARAMS, stride)
    assert np.array_equal(sc2, sc) and np.array_equal(sp2, sp) and np.array_equal(cnt2, cnt) and np.array_equal(ops2, ops)
    for k in range(0, n, 50):
        a, b = h1[k * L:(k + 1) * L], h2[k * L:(k + 1) * L]
        want = BO.gotoh_banded_span(a, b, lo, hi)
        assert (int(sc[k]),) + tuple(int(x) for x in sp[k]) == want, k
        assert check_cigar(api.cigar_string(ops[k, :cnt[k]]), a, b, sp[k], api.DEFAULT_PARAMS, lo, hi) == (want[0], True, True), k


@pytest.mark.parametrize("W", [128, 512])
def test_ops_overflow(W):
    import re
    from concurrentproject_b200 import api
    s1, s2 = _mixed_pairs(1400 + W, 40)
    p, lo, hi = (2, -3, 5, 1), -W // 2, W // 2 - 1
    full = api.align_banded_batch(s1, s2, lo, hi, p, ops_stride=20000)
    nops = [len(re.findall(r"\d+[=XID]", c)) for c in full[2]]
    f1, o1, l1 = api._flatten(s1)
    f2, o2, l2 = api._flatten(s2)
    scores, spans, ops, cnt = api.align_banded_batch_ops(f1, o1, l1, f2, o2, l2, lo, hi, p, ops_stride=5)
    assert any(x > 5 for x in nops) and any(0 < x <= 5 for x in nops)
    assert np.array_equal(scores, full[0]) and np.array_equal(spans, full[1])
    for k, x in enumerate(nops):
        if x > 5:
            assert cnt[k] == -x and not ops[k].any()
        else:
            assert cnt[k] == x and api.cigar_string(ops[k, :cnt[k]]) == full[2][k]


def test_errors():
    """Widths other than 64 / 128 / 256 / 512 are refused by every call; score and align refuse the same inputs."""
    from concurrentproject_b200 import api
    good1, good2 = [b"ACGT" * 10, b"ACG"], [b"ACGA" * 12, b"TTACG"]
    cases = [(good1, good2, -48, 47, O.DEFAULT),                                   # 96 diagonals
             (good1, good2, -96, 95, O.DEFAULT),                                   # 192
             (good1, good2, -512, 511, O.DEFAULT),                                 # 1024
             (good1 + [b"ACNGT"], good2 + [b"ACGT"], -128, 127, O.DEFAULT),       # alphabet
             (good1 + [b"A" * 800], good2 + [b"A" * 900], -256, 255, (50, -1, 1, 1))]   # match * min(len) out of range
    for s1, s2, lo, hi, p in cases:
        with pytest.raises(api.SwbError) as e1:
            api.score_banded_batch(s1, s2, lo, hi, p)
        with pytest.raises(api.SwbError) as e2:
            api.align_banded_batch(s1, s2, lo, hi, p)
        assert e1.value.code == e2.value.code, (lo, hi, e1.value, e2.value)
    for w in (65, 73, 96, 100, 192, 1024):
        assert _single(b"ACGT", b"ACGT", 0, w - 1, O.DEFAULT)[0] == -2
        with pytest.raises(api.SwbError) as e:
            api.score_banded_batch(good1, good2, 0, w - 1)
        assert e.value.code == -2


def test_two_gpus_identical():
    import torch
    from concurrentproject_b200 import api
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s1, s2 = _drift_pairs(1500, 120, 256)
    p = (2, -3, 5, 1)
    one = (api.score_banded_batch(s1, s2, -128, 127, p), api.align_banded_batch(s1, s2, -256, 255, p))
    api.set_devices(2)
    try:
        two = (api.score_banded_batch(s1, s2, -128, 127, p), api.align_banded_batch(s1, s2, -256, 255, p))
    finally:
        api.set_devices(1)
    assert np.array_equal(one[0], two[0])
    assert np.array_equal(one[1][0], two[1][0]) and np.array_equal(one[1][1], two[1][1]) and one[1][2] == two[1][2]
