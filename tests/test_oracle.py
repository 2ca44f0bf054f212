"""Pins the CPU oracle (oracle/gotoh_oracle.c) to the reference: its known-answer tables, its 30
recorded seeded scores, fixtures produced by the unmodified reference build, and the reference's scores on fresh random
inputs (stored in tests/golden/ref_scores_live.json, and live when oracle/_ref/libref.so is present)."""
import numpy as np
import pytest

import oracle_lib as O
from conftest import GOLDEN, fixture_pair, load_json, mt_pairs
from concurrentproject_b200 import rng

ALL = (O.gotoh_full, O.gotoh_rolling, O.lazy_smith, O.gotoh_mt)


def test_rng_python_matches_c():
    for seed, stream, n in [(1, 0, 0), (1, 0, 1), (2, 5, 31), (2, 5, 32), (3, 9, 33), (99, 12345678901, 1000)]:
        assert bytes(rng.random_acgt(seed, stream, n)) == bytes(O.random_acgt(seed, stream, n))
    lib = O.oracle()
    for idx in [0, 1, 2**31, 2**40 + 17]:
        assert int(rng.mix64(7, 3, idx)) == lib.oracle_mix64(7, 3, idx)


def test_known_answer_tables():
    for c in load_json("kat.json"):
        for f in ALL:
            assert f(c["seq1"], c["seq2"]) == c["score"], (f.__name__, c["source"])
        # SmithDiagonalGPU's linear-gap recurrence equals affine because G_INIT == G_EXT
        assert O.linear_gap(c["seq1"], c["seq2"]) == c["score"], c["source"]


@pytest.mark.parametrize("L", [32, 516, 4096])
def test_reference_recorded_seeded_scores(L):
    # cudaSmithM.cu:285-294 / 314-323 / 342-351
    for a, b, want in mt_pairs(L):
        assert O.gotoh_rolling(a, b) == want
        assert O.lazy_smith(a, b) == want
        if L <= 516:
            assert O.gotoh_full(a, b) == want
        assert O.gotoh_mt(a, b, threads=3) == want


def test_reference_fixture_scores_default_params():
    for c in load_json("ref_scores_default.json"):
        if c["n"] > 20000:
            continue  # cfg2 full size: covered by the gpu suite and test_oracle_cfg2_slow
        a, b = fixture_pair(c)
        assert O.gotoh_rolling(a, b) == c["score"], c
        if c["n"] * c["m"] <= 4_000_000:
            assert O.gotoh_full(a, b) == c["score"], c
            assert O.lazy_smith(a, b) == c["score"], c
        assert O.gotoh_mt(a, b, threads=4) == c["score"], c


def test_reference_fixture_scores_other_params():
    ndiff = 0
    for c in load_json("ref_scores_params.json"):
        a, b = fixture_pair(c)
        p = tuple(c["params"])
        assert O.gotoh_full(a, b, p) == c["score_main"], c      # contract: main.cpp
        assert O.gotoh_rolling(a, b, p) == c["score_main"], c
        assert O.gotoh_mt(a, b, p, threads=2) == c["score_main"], c
        assert O.lazy_smith(a, b, p) == c["score_lazy"], c       # restated incl. its G_INIT>2*G_EXT over-score
        ndiff += c["score_main"] != c["score_lazy"]
    assert ndiff > 0  # the divergence regime is represented in the fixtures


def test_argument_swap_symmetry_and_edges():
    for k in range(40):
        n, m = int(rng.mix64(5, 1, k) % 90), int(rng.mix64(5, 2, k) % 90)
        a, b = rng.random_acgt(5, 2 * k, n), rng.random_acgt(5, 2 * k + 1, m)
        s = O.gotoh_full(a, b)
        assert s == O.gotoh_full(b, a) == O.gotoh_rolling(a, b) == O.gotoh_mt(a, b, threads=2)
    assert O.gotoh_rolling(b"", b"") == 0
    assert O.gotoh_rolling(b"ACGT" * 10, b"ACGT" * 10) == 40


def _banded_bruteforce(a, b, lo, hi, p=O.DEFAULT):
    ma, mi, gi, ge = p
    n, m = len(a), len(b)
    H = np.zeros((m + 1, n + 1), dtype=np.int64); E = H.copy(); F = H.copy()
    best = 0; cells = 0
    for i in range(1, m + 1):
        for j in range(1, n + 1):
            if not (lo <= j - i <= hi):
                continue
            cells += 1
            E[i][j] = max(E[i][j - 1] - ge, H[i][j - 1] - gi)
            F[i][j] = max(F[i - 1][j] - ge, H[i - 1][j] - gi)
            H[i][j] = max(0, H[i - 1][j - 1] + (ma if a[j - 1] == b[i - 1] else mi), E[i][j], F[i][j])
            best = max(best, int(H[i][j]))
    return best, cells


def test_banded_oracle_against_masked_full_matrix():
    for k, (n, m, lo, hi) in enumerate([(40, 40, -32, 31), (70, 90, -32, 31), (90, 70, -32, 31), (50, 50, -3, 2),
                                         (30, 64, -5, 40), (64, 30, -40, 5), (20, 20, -100, 100), (33, 35, 0, 0), (10, 60, -32, 31)]):
        a = rng.random_acgt(21, k, n)
        b = rng.mutate(a, 21, 100 + k, 0.1, 0.05)[:m] if k % 2 == 0 else rng.random_acgt(21, 50 + k, m)
        for p in (O.DEFAULT, (2, -3, 5, 1)):
            want, cells = _banded_bruteforce(bytes(a), bytes(b), lo, hi, p)
            got, gcells = O.gotoh_banded(a, b, lo, hi, p, want_cells=True)
            assert (got, gcells) == (want, cells), (n, m, lo, hi, p)
    a = rng.random_acgt(22, 0, 300); b = rng.random_acgt(22, 1, 280)
    assert O.gotoh_banded(a, b, -10**6, 10**6) == O.gotoh_rolling(a, b)


def test_batch_entry_points():
    s1 = [rng.random_acgt(31, k, 20 + 7 * k) for k in range(9)] + [np.zeros(0, np.uint8)]
    s2 = [rng.random_acgt(32, k, 90 - 5 * k) for k in range(9)] + [rng.random_acgt(32, 99, 5)]
    got = O.gotoh_batch(s1, s2, threads=3)
    assert list(got) == [O.gotoh_rolling(a, b) for a, b in zip(s1, s2)]
    gb = O.gotoh_banded_batch(s1, s2, -8, 7, threads=2)
    assert list(gb) == [O.gotoh_banded(a, b, -8, 7) for a, b in zip(s1, s2)]


@pytest.mark.skipif(not (GOLDEN / "ref_scores_live.json").exists() and not O.ref_available(),
                    reason="needs the original project's scores: tests/golden/ref_scores_live.json (written by "
                           "tests/golden/make_golden.py --live) or oracle/_ref/libref.so")
def test_oracle_equals_live_reference_on_fresh_inputs():
    """The reference's three CPU functions on 25 fresh seeded pairs: the stored scores when they are committed, and the
    reference itself when oracle/_ref/libref.so is built."""
    from golden.make_golden import fresh_inputs
    pairs = list(fresh_inputs())
    sources = []
    if (GOLDEN / "ref_scores_live.json").exists():
        sources.append(load_json("ref_scores_live.json")["fresh"])
    if O.ref_available():
        fns = ("ref_SmithWatermanScore", "ref_LazySmith", "ref_ParallelLazySmith_threads")
        sources.append([[O.ref_call(f, a, b) for f in fns] for a, b in pairs])
    for scores in sources:
        assert len(scores) == len(pairs)
        for k, ((a, b), three) in enumerate(zip(pairs, scores)):
            want = three[0]
            assert three == [want] * 3, k
            assert O.gotoh_rolling(a, b) == want and O.gotoh_full(a, b) == want and O.lazy_smith(a, b) == want, k


def test_end_cell_and_span_oracles_are_self_consistent():
    """oracle_gotoh_end / oracle_gotoh_span (new semantics, no reference counterpart): the score equals main.cpp's, the
    end cell holds the maximum and is the first one in (j, i) order, the span's sub-rectangle scores the same and its
    corner cells are aligned matches."""
    r = np.random.default_rng(123)
    for trial in range(60):
        n, m = int(r.integers(1, 90)), int(r.integers(1, 90))
        k = int(r.integers(2, 5))
        a = r.integers(0, k, n, dtype=np.uint8) + 65
        b = r.integers(0, k, m, dtype=np.uint8) + 65
        p = [(1, -1, 1, 1), (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (1, -1, 0, 0), (4, -1, 2, 5)][trial % 6]
        s = O.gotoh_full(a, b, p)
        se, ie, je = O.gotoh_end(a, b, p)
        assert se == s
        sp = O.gotoh_span(a, b, p)
        assert sp[0] == s and sp[3:] == (ie, je)
        if s == 0:
            assert sp == (0, 0, 0, 0, 0)
            continue
        i0, j0 = sp[1], sp[2]
        assert 1 <= i0 <= ie <= m and 1 <= j0 <= je <= n
        assert O.gotoh_full(a[j0 - 1:je], b[i0 - 1:ie], p) == s
        assert a[je - 1] == b[ie - 1] and a[j0 - 1] == b[i0 - 1]          # a best alignment starts and ends on a match
        # no cell with the maximum lies before the end cell in (j, i) order: prefixes that stop short of it score less
        if je > 1:
            assert O.gotoh_full(a[:je - 1], b, p) < s
        if ie > 1:
            assert O.gotoh_full(a[:je], b[:ie - 1], p) < s


def test_fast_oracle_equals_the_rolling_row_oracle():
    """oracle/gotoh_fast.c (one tile per SIMD lane; pins the scores under tests/golden/large_scores.json) against
    oracle_gotoh_rolling on ragged tile edges, non-default parameters, and a pair larger than one tile diagonal."""
    for (n, m, seed) in [(1, 1, 1), (3, 700, 2), (255, 257, 3), (256, 256, 4), (1000, 1000, 5), (5000, 3333, 6), (4097, 8191, 7)]:
        a = rng.random_acgt(seed, 0, n)
        b = rng.mutate(rng.random_acgt(seed, 0, m) if m <= n else rng.random_acgt(seed, 1, m), seed, 3, 0.1, 0.05)
        for p in [(1, -1, 1, 1), (2, -3, 5, 1), (5, -4, 11, 1), (1, -1, 0, 0)]:
            assert O.gotoh_fast(a, b, p) == O.gotoh_rolling(a, b, p), (n, m, p)
    a = rng.random_acgt(11, 0, 30000)
    b = rng.mutate(a, 11, 1, 0.15, 0.05)[:20001]
    assert O.gotoh_fast(a, b) == O.gotoh_mt(a, b)
    assert O.gotoh_fast(b"", b"ACGT") == 0


def test_pinned_large_scores_file():
    """The committed pins: cfg2 agrees with the unmodified reference's own LazySmith (ref_scores_default.json), the
    small one is recomputed here."""
    big = load_json("large_scores.json")
    assert {"cfg2", "ring400k", "n1m", "cfg3"} <= set(big)
    ref = [c for c in load_json("ref_scores_default.json") if c.get("config") == "cfg2"][0]
    assert big["cfg2"]["score"] == ref["score"]
    c = big["cfg2"]
    assert O.gotoh_fast(rng.random_acgt(c["seed"], 0, c["n"]), rng.random_acgt(c["seed"], 1, c["m"])) == c["score"]
