"""Long-pair batch alignment (csrc/swb_align_long.cuh) without a GPU: the per-pair warp bodies run on CPU threads
(tests/emu/align_long_emu.cu, one pthread per lane, two warps drawing pairs from a counter, the host driver's trace
rounds) against the pure-Python reference of the batch alignment contract in test_align_batch_emu.py, which is pinned to
the C oracle's score and span on every case.  Needs nvcc (host compile only)."""
import re
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng
from test_align_batch_emu import OPS, PARAMS, ref_align, rescore

EMU_DIR = Path(__file__).resolve().parent / "emu"
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    exe = EMU_DIR / "align_long_emu"
    src = EMU_DIR / "align_long_emu.cu"
    hdrs = [EMU_DIR.parent.parent / "concurrentproject_b200" / "csrc" / h
            for h in ("swb_align_long.cuh", "swb_align_banded.cuh", "swb_align_batch.cuh", "swb_device.cuh")]
    if not exe.exists() or exe.stat().st_mtime < max(x.stat().st_mtime for x in [src] + hdrs):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(src),
                        "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("align_long_emu")

    def run(s1, s2, p, slot_words=1 << 22, pool_words=0, ops_stride=None):
        if ops_stride is None:
            ops_stride = max(1, max(len(a) + len(b) for a, b in zip(s1, s2)))
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(exe), str(f), *map(str, [*p, slot_words, pool_words, ops_stride])], capture_output=True,
                             text=True, timeout=1800, check=True).stdout.strip().split("\n")
        rows = []
        for line in res[:-1]:
            v = [int(x) for x in line.split()]
            rows.append((v[0], tuple(v[1:5]), v[5], [(OPS[w & 15], w >> 4) for w in v[6:]]))
        rounds, err = re.fullmatch(r"rounds (\d+) err (\d+) cells \d+", res[-1]).groups()
        return rows, int(rounds), int(err)
    return run


def _check(rows, s1, s2, p):
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align(a, b, p)
        assert (want[0],) + want[1] == O.gotoh_span(a, b, p), (k, p)            # the reference is the oracle's score and span
        score, span, n, runs = rows[k]
        assert (score, span, runs) == want, (k, len(a), len(b), p, score, span, runs[:8], want[0], want[1], want[2][:8])
        assert n == len(runs)
        if score > 0:
            assert rescore(runs, a, b, span, p) == score, (k, p)


def _planted(seed, k, short, extra, sub=0.04, indel=0.02):
    """A window of short + extra bases and a mutated copy of its middle cut to `short` bases (random if k % 3 == 2)."""
    w = bytes(rng.random_acgt(seed, 2 * k, short + extra))
    if k % 3 == 2 or short < 8:
        return bytes(rng.random_acgt(seed, 2 * k + 1, short)), w
    o = extra // 2
    rd = bytes(rng.mutate(np.frombuffer(w[o:o + short], np.uint8), seed, 2 * k + 1, sub, indel))[:short]
    if len(rd) < short:
        rd += bytes(rng.random_acgt(seed, 2 * k + 3, short - len(rd)))
    return rd, w


def _ragged(seed, npairs, max_short=300, max_extra=300):
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(npairs):
        a, b = _planted(seed, k, int(r.integers(0, max_short + 1)), int(r.integers(0, max_extra + 1)))
        if k % 2:
            a, b = b, a                                      # both orientations of the packer
        s1.append(a); s2.append(b)
    return s1, s2


@pytest.mark.parametrize("p", PARAMS)
def test_align_long_kernel_bodies(emu, p):
    """17 ragged pairs (short sides 0..300, so some cross the 256-row band edge; planted and random; both orientations)."""
    s1, s2 = _ragged(170 + PARAMS.index(p), 17)
    rows, rounds, err = emu(s1, s2, p)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, p)


@pytest.mark.parametrize("p", [O.DEFAULT, (2, -3, 5, 1)])
def test_band_edges(emu, p):
    """Short sides at and next to every band edge up to five bands, in both orientations: the hand-off through the
    boundary row, the last band's pad rows and a walk that leaves its staged lines and the band together."""
    s1, s2 = [], []
    for k, short in enumerate((1, 255, 256, 257, 511, 512, 513, 1025)):
        q, t = _planted(300 + PARAMS.index(p) if p in PARAMS else 300, k, short, 24 + 7 * k)
        s1 += [q, t]; s2 += [t, q]
    rows, rounds, err = emu(s1, s2, p)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, p)


def _acfill(seed, k, n):
    """n bases of A / C only (never equal to the G / T fillers below)"""
    return bytes(b"AC"[(c >> 1) & 1] for c in rng.random_acgt(seed, k, n))


def test_tie_rules_across_bands(emu):
    """Equal maxima in two bands, and ties that differ only in row or only in column.  Patterns of A / C sit in fillers
    that never match (G in one sequence, T in the other), so each planted copy scores exactly len * match.  Each case
    runs in both orientations: seq1 as the shorter sequence (rows) and as the longer (columns)."""
    A, B = _acfill(7, 0, 40), _acfill(7, 1, 40)
    cases = [
        # A at rows 11.. and B at rows 301..; B at columns 51.., A at columns 601..: the later band holds the smaller column
        (b"G" * 10 + A + b"G" * 250 + B + b"G" * 30, b"T" * 50 + B + b"T" * 510 + A + b"T" * 40),
        # one column, two rows in two bands
        (b"G" * 10 + A + b"G" * 250 + A + b"G" * 30, b"T" * 600 + A + b"T" * 40),
        # one row, two columns
        (b"G" * 270 + A + b"G" * 30, b"T" * 100 + A + b"T" * 460 + A + b"T" * 40),
        # equal maxima in two bands at the same column distance
        (b"G" * 200 + A + b"G" * 20 + A + b"G" * 30, b"T" * 300 + A + b"T" * 300),
    ]
    s1, s2 = [], []
    for q, t in cases:
        s1 += [q, t]; s2 += [t, q]
    for p in (O.DEFAULT, (2, -3, 5, 1), (1, -1, 0, 0)):
        rows, _, err = emu(s1, s2, p)
        assert err == 0
        _check(rows, s1, s2, p)


def test_gap_across_band_edge(emu):
    """A run of 30 extra bases of the shorter sequence across row 256 (a gap along the rows: E when the shorter sequence
    is seq1, F when it is seq2), and a run of 30 extra bases of the longer sequence near that edge."""
    x = bytes(rng.random_acgt(11, 0, 700))
    ins = bytes(rng.random_acgt(11, 1, 30))
    q1, t1 = x[:240] + ins + x[240:480], x[:600]
    q2, t2 = x[:250] + x[280:530], x[:600]
    s1, s2 = [q1, t1, q2, t2], [t1, q1, t2, q2]
    for p in ((2, -3, 5, 1), (1, -1, 1, 1), (2, -1, 1, 3)):
        rows, _, err = emu(s1, s2, p)
        assert err == 0
        _check(rows, s1, s2, p)


def test_zero_scores_and_empty(emu):
    s1 = [b"", b"ACGT", b"A" * 300, b"G" * 40, b"C"]
    s2 = [b"ACGT", b"", b"C" * 500, b"T" * 700, b"C"]
    for p in (O.DEFAULT, (2, -1, 1, 3)):
        rows, _, err = emu(s1, s2, p)
        assert err == 0
        assert [r[0] for r in rows[:4]] == [0, 0, 0, 0]
        _check(rows, s1, s2, p)


def test_pool_and_pending_rounds(emu):
    """Slots too small for any span and a pool with room for about the largest one: every pair takes a piece of the
    pool or waits for a later round, and the results do not change."""
    s1, s2 = _ragged(191, 10, max_short=280, max_extra=120)
    for p in (O.DEFAULT, (2, -3, 5, 1)):
        rows, rounds, err = emu(s1, s2, p, slot_words=4, pool_words=1)
        assert err == 0 and rounds > 1
        _check(rows, s1, s2, p)


def test_ops_stride_overflow(emu):
    """ops_count = -(operations) where ops_stride is too small, nothing written; the other pairs complete."""
    s1, s2 = _ragged(192, 10, max_short=280, max_extra=120)
    p = (2, -3, 5, 1)
    rows, _, err = emu(s1, s2, p, ops_stride=3)
    assert err == 0
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align(a, b, p)
        score, span, n, runs = rows[k]
        assert (score, span) == (want[0], want[1])
        if len(want[2]) > 3:
            assert n == -len(want[2]) and runs == []
        else:
            assert n == len(want[2]) and runs == want[2]
