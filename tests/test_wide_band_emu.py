"""Bands of 128, 256 and 512 diagonals without a GPU: the product's banded score body (banded_warpS<MODE, 8, W>) and
alignment bodies (band_span_pair<K>, band_trace_pair<K>) run on CPU threads (tests/emu/wide_band_emu.cu, one pthread per
lane of two emulated warps) against the C checkers (oracle_gotoh_banded_batch, oracle_gotoh_banded_span) and the
Python reference of the banded alignment contract.  Needs nvcc (host compile only)."""
import re
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import banded_oracle as BO
import oracle_lib as O
from concurrentproject_b200 import rng
from test_align_banded_emu import _pairs, path_in_band, ref_align_banded
from test_align_batch_emu import ref_align, rescore

EMU_DIR = Path(__file__).resolve().parent / "emu"
OPS = {1: "I", 2: "D", 7: "=", 8: "X"}
# five parameter sets: linear and affine, gap_ext > gap_init among them; MODE 1 (linear kernel) where gap_init == gap_ext
PARAMS = [O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (5, -4, 11, 1)]
WIDTHS = [128, 256, 512]
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    work = tmp_path_factory.mktemp("wide_band_emu")
    exe = work / "wide_band_emu"
    subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe),
                    str(EMU_DIR / "wide_band_emu.cu"), "-lpthread"], check=True)

    def write(s1, s2):
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        return f

    def score(s1, s2, W, p, lo, mode=None):
        if mode is None:
            mode = 1 if p[2] == p[3] else 0
        out = subprocess.run([str(exe), "score", str(write(s1, s2)), *map(str, [W, mode, lo, *p])], capture_output=True,
                             text=True, timeout=900, check=True).stdout
        return [int(x) for x in out.split()[1:]]

    def align(s1, s2, W, p, lo, slot_words=1 << 16, pool_words=0, ops_stride=None):
        if ops_stride is None:
            ops_stride = max(1, max(len(a) + len(b) for a, b in zip(s1, s2)))
        res = subprocess.run([str(exe), "align", str(write(s1, s2)), *map(str, [W, lo, *p, slot_words, pool_words, ops_stride])],
                             capture_output=True, text=True, timeout=900, check=True).stdout.strip().split("\n")
        rows = []
        for line in res[:-1]:
            v = [int(x) for x in line.split()]
            rows.append((v[0], tuple(v[1:5]), v[5], [(OPS[w & 15], w >> 4) for w in v[6:]]))
        rounds, err = re.fullmatch(r"rounds (\d+) err (\d+) cells \d+", res[-1]).groups()
        return rows, int(rounds), int(err)

    class E:
        pass
    e = E()
    e.score, e.align = score, align
    return e


def _score_pairs(seed, npairs, max_len):
    """Ragged pairs, related (a mutated copy, 8 % substitutions, 3 % indels) and unrelated."""
    r = np.random.default_rng(seed)
    a = [bytes(rng.random_acgt(seed, k, int(r.integers(1, max_len)))) for k in range(npairs)]
    b = [bytes(rng.mutate(np.frombuffer(x, np.uint8), seed, 100 + k, 0.08, 0.03)) if k % 3 else
         bytes(rng.random_acgt(seed + 1, k, int(r.integers(1, max_len)))) for k, x in enumerate(a)]
    return a, b


def _planted_indel(seed, n, indel):
    """seq2 = seq1 with `indel` bases deleted in the middle (a few substitutions around): the best alignment leaves the
    main diagonal by `indel` diagonals."""
    a = rng.random_acgt(seed, 0, n)
    b = np.concatenate([a[:n // 2], a[n // 2 + indel:]])
    b = rng.mutate(b, seed, 1, 0.02, 0.0)
    return bytes(a), bytes(b)


# ---- score body -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W", WIDTHS)
def test_wide_score_body(emu, W):
    """Five parameter sets in both recurrences (linear where gap_init == gap_ext, affine always), centred and shifted bands;
    a pair count that leaves the last group of a warp partly empty (W = 128: 4 pairs a warp, W = 256: 2)."""
    a, b = _score_pairs(70 + W, {128: 11, 256: 7, 512: 5}[W], 700)
    for lo in (-W // 2, -W // 2 + 7, -10, -W + 3, 20):
        for p in PARAMS:
            modes = (0, 1) if p[2] == p[3] else (0,)
            for mode in modes:
                want = O.gotoh_banded_batch(a, b, lo, lo + W - 1, p).tolist()
                assert emu.score(a, b, W, p, lo, mode) == want, (W, lo, p, mode)


@pytest.mark.parametrize("W", WIDTHS)
def test_wide_score_band_offsets(emu, W):
    """band_lo of both parities and all 32 residues mod 32: the first chunk's ring contents and the column window's bit
    offset follow band_lo."""
    a, b = _score_pairs(80 + W, 4, 600)
    for r in range(32):
        lo = -W // 2 - 16 + r
        p = PARAMS[r % len(PARAMS)]
        want = O.gotoh_banded_batch(a, b, lo, lo + W - 1, p).tolist()
        assert emu.score(a, b, W, p, lo) == want, (W, lo, p)


@pytest.mark.parametrize("W", WIDTHS)
def test_wide_score_band_edges(emu, W):
    """Bands that start outside the matrix, that miss it (score 0), and pairs shorter than the band (the full score)."""
    a, b = _score_pairs(90 + W, 6, 200)
    for lo in (250, -(W + 260), 190, -(W + 150), -W + 1, 0):
        for p in (O.DEFAULT, (2, -3, 5, 1)):
            want = O.gotoh_banded_batch(a, b, lo, lo + W - 1, p).tolist()
            assert emu.score(a, b, W, p, lo) == want, (W, lo, p)
    got = emu.score(a, b, W, O.DEFAULT, 250)
    assert got == [0] * len(a)
    short_a = [x[:W // 4] for x in a]
    short_b = [x[:W // 4] for x in b]
    for p in PARAMS:
        assert emu.score(short_a, short_b, W, p, -W // 2) == [O.gotoh_full(x, y, p) for x, y in zip(short_a, short_b)]


def test_planted_indel_score(emu):
    """An 80-100 base deletion moves the best alignment beyond 32 diagonals: W = 64 scores less, W = 256 recovers the
    unbanded score."""
    for k, indel in enumerate((80, 93, 100)):
        a, b = _planted_indel(200 + k, 900, indel)
        full = O.gotoh_full(a, b)
        assert O.gotoh_banded(a, b, -32, 31) < full
        assert emu.score([a], [b], 256, O.DEFAULT, -128) == [full]
        assert emu.score([a], [b], 512, (2, -3, 5, 1), -256) == [O.gotoh_full(a, b, (2, -3, 5, 1))]


# ---- alignment bodies -----------------------------------------------------------------------------------------------
def _check(rows, s1, s2, p, lo, hi):
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align_banded(a, b, p, lo, hi)
        score, span, n, runs = rows[k]
        assert (score, span, runs) == want, (k, p, lo, score, span, runs[:8], want[0], want[1], want[2][:8])
        assert n == len(runs)
        if score > 0:
            assert rescore(runs, a, b, span, p) == score and path_in_band(runs, span, lo, hi), (k, p, lo)


@pytest.mark.parametrize("W", WIDTHS)
def test_wide_align_bodies(emu, W):
    """Ragged pairs (related and unrelated, both orientations) under a centred band and bands above / below the main
    diagonal, five parameter sets; 5 pairs over 2 warps leave the last warp's turn partly empty."""
    for p in PARAMS:
        s1, s2 = _pairs(300 + W + PARAMS.index(p), 5, max_len=160)
        rows, rounds, err = emu.align(s1, s2, W, p, -W // 2)
        assert err == 0 and rounds == 1
        _check(rows, s1, s2, p, -W // 2, W // 2 - 1)
    for shift, lo in ((40, 20 - W // 2), (-40, -60 - W // 2), (30, 3)):
        s1, s2 = _pairs(310 + W, 4, max_len=200, shift=shift)
        rows, _, err = emu.align(s1, s2, W, (2, -3, 5, 1), lo)
        assert err == 0
        _check(rows, s1, s2, (2, -3, 5, 1), lo, lo + W - 1)


@pytest.mark.parametrize("W", WIDTHS)
def test_wide_align_edges(emu, W):
    """Bands that cut row 1 / column 1 or hold no cell (score 0), both parities of band_lo, and pairs shorter than the
    band, which give the read-batch call's span and CIGAR."""
    x = bytes(rng.random_acgt(19, 0, 120))
    for s1, s2, p, lo in [([x], [x], O.DEFAULT, 3), ([x], [x], O.DEFAULT, -W + 5), ([x], [x], (2, -1, 1, 3), -W + 4),
                          ([x[:30]], [x[:30]], O.DEFAULT, 40), ([x[:30]], [x[:30]], O.DEFAULT, -W - 40),
                          ([b""], [x], O.DEFAULT, -W // 2), ([x], [b""], O.DEFAULT, -W // 2)]:
        rows, _, err = emu.align(s1, s2, W, p, lo)
        assert err == 0
        _check(rows, s1, s2, p, lo, lo + W - 1)
    s1, s2 = _pairs(320 + W, 6, max_len=W // 4)
    for p in PARAMS:
        rows, _, err = emu.align(s1, s2, W, p, -W // 2 + 1)
        assert err == 0
        for k, (a, b) in enumerate(zip(s1, s2)):
            score, span, n, runs = rows[k]
            assert (score, span, runs) == ref_align(a, b, p), (W, p, k)


@pytest.mark.parametrize("W", WIDTHS)
def test_wide_align_planted_indel(emu, W):
    """A planted 80-100 base deletion: the span the emulated warps find equals oracle_gotoh_banded_span, the CIGAR
    re-scores to the score with every cell in the band, and from W = 256 on the score is the unbanded one."""
    for k, indel in enumerate((80, 100)):
        a, b = _planted_indel(400 + k, 500, indel)
        for p in (O.DEFAULT, (2, -3, 5, 1)):
            lo = -W // 2
            rows, _, err = emu.align([a], [b], W, p, lo)
            assert err == 0
            score, span, n, runs = rows[0]
            assert (score,) + span == BO.gotoh_banded_span(a, b, lo, lo + W - 1, p)
            assert score == O.gotoh_banded(a, b, lo, lo + W - 1, p)
            assert rescore(runs, a, b, span, p) == score and path_in_band(runs, span, lo, lo + W - 1)
            if W >= 256:
                assert score == O.gotoh_full(a, b, p) > O.gotoh_banded(a, b, -32, 31, p)


@pytest.mark.parametrize("W", [128, 512])
def test_wide_align_pool_and_overflow(emu, W):
    """Slots too small for any span (the pool and pending rounds), and ops_stride too small (ops_count = -operations)."""
    s1, s2 = _pairs(330 + W, 6, max_len=120)
    p = (2, -3, 5, 1)
    rows, rounds, err = emu.align(s1, s2, W, p, -W // 2, slot_words=4, pool_words=1)
    assert err == 0 and rounds > 1
    _check(rows, s1, s2, p, -W // 2, W // 2 - 1)
    rows, _, err = emu.align(s1, s2, W, p, -W // 2, ops_stride=3)
    assert err == 0
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align_banded(a, b, p, -W // 2, W // 2 - 1)
        score, span, n, runs = rows[k]
        assert (score, span) == (want[0], want[1])
        assert (n, runs) == ((-len(want[2]), []) if len(want[2]) > 3 else (len(want[2]), want[2]))
