"""Byte batches (csrc/swb_align_batch.cuh with align_code<8>, csrc/swb_bytes_batch.cu) without a GPU: the per-pair kernel
bodies of the byte score, span and trace kernels run on CPU threads (tests/emu/bytes_batch_emu.cu, one pthread per lane of
an emulated warp, the host driver's trace rounds) on pairs in any bytes, against the C oracle's score and span on the raw
bytes and the Python reference of the batch-alignment contract (test_align_batch_emu.ref_align).  On A,C,G,T input the
byte bodies give exactly what the 2-bit bodies give.  Needs nvcc (host compile only)."""
import re
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng
from test_align_batch_emu import ref_align, rescore

EMU_DIR = Path(__file__).resolve().parent / "emu"
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")

PARAMS = [O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (1, -1, 0, 0), (5, -4, 11, 1)]
OPS = {1: "I", 2: "D", 7: "=", 8: "X"}
ALPHABETS = {
    "acgtn": b"ACGTN",
    "iupac": b"ACGTRYSWKMBDHVN",
    "protein": b"ACDEFGHIKLMNPQRSTVWY",
    "all256": bytes(range(256)),
}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    exe = tmp_path_factory.mktemp("bytes_batch_bin") / "bytes_batch_emu"
    src = EMU_DIR / "bytes_batch_emu.cu"
    subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(src),
                    "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("bytes_batch_emu")

    def run(s1, s2, p, bits=8, slot_words=4096, pool_words=0, ops_stride=None):
        if ops_stride is None:
            ops_stride = max(1, max(len(a) + len(b) for a, b in zip(s1, s2)))
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(exe), str(f), str(bits), *map(str, [*p, slot_words, pool_words, ops_stride])],
                             capture_output=True, text=True, timeout=900, check=True).stdout.strip().split("\n")
        rows = []
        for line in res[:-1]:
            v = [int(x) for x in line.split()]
            rows.append((v[0], v[1], tuple(v[2:6]), v[6], [(OPS[w & 15], w >> 4) for w in v[7:]]))
        rounds, err = re.fullmatch(r"rounds (\d+) err (\d+)", res[-1]).groups()
        return rows, int(rounds), int(err)
    return run


def _draw(r, alphabet, n):
    return bytes(np.frombuffer(alphabet, np.uint8)[r.integers(0, len(alphabet), size=n)].tobytes())


def _mutate(r, alphabet, s, sub=0.08, indel=0.03):
    out = bytearray()
    for c in s:
        u = r.random()
        if u < indel / 2:
            continue                                              # deletion
        if u < indel:
            out += _draw(r, alphabet, 1)                          # insertion before c
        out.append(_draw(r, alphabet, 1)[0] if r.random() < sub else c)
    return bytes(out)


def _pairs(seed, alphabet, npairs, max_read=90, max_win=220):
    """Ragged pairs over `alphabet`: half a read planted in its window with substitutions and indels, half unrelated;
    every third pair with the read as seq2 (both orientations of the packer)."""
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(npairs):
        w = _draw(r, alphabet, int(r.integers(1, max_win + 1)))
        rl = int(r.integers(0, max_read + 1))
        if k % 2 == 0 and len(w) > rl > 4:
            o = int(r.integers(0, len(w) - rl))
            rd = _mutate(r, alphabet, w[o:o + rl])
        else:
            rd = _draw(r, alphabet, rl)
        if k % 3 == 1:
            s1.append(w); s2.append(rd)
        else:
            s1.append(rd); s2.append(w)
    return s1, s2


def _check(rows, s1, s2, p):
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align(a, b, p)
        assert (want[0],) + want[1] == O.gotoh_span(a, b, p), (k, p)            # the reference is the oracle's score and span
        score_only, score, span, n, runs = rows[k]
        assert score_only == score == O.gotoh_rolling(a, b, p), (k, p, score_only, score)
        assert (score, span, runs) == want, (k, p, score, span, runs[:8], want[0], want[1], want[2][:8])
        assert n == len(runs)
        if score > 0:
            assert rescore(runs, a, b, span, p) == score, (k, p)


@pytest.mark.parametrize("name", list(ALPHABETS))
def test_alphabets(emu, name):
    """ACGT+N, IUPAC codes, a 20-letter protein alphabet and all 256 byte values: score-only pass, span and CIGAR."""
    s1, s2 = _pairs(300 + len(name), ALPHABETS[name], 33)
    rows, rounds, err = emu(s1, s2, O.DEFAULT)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, O.DEFAULT)


@pytest.mark.parametrize("p", PARAMS)
def test_parameter_sets(emu, p):
    """Six parameter sets (gap_ext > gap_init among them), each on a different alphabet."""
    name = list(ALPHABETS)[PARAMS.index(p) % len(ALPHABETS)]
    s1, s2 = _pairs(400 + PARAMS.index(p), ALPHABETS[name], 25)
    rows, rounds, err = emu(s1, s2, p)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, p)


def test_bytes_no_byte_can_take_the_pad_code(emu):
    """0x04 (the 2-bit layout's pad code), 0x00 and 0xFF at the ends of both sequences, in both orientations and against
    each other: columns past the end of T never match a byte, so no score reaches past the sequence."""
    cases = []
    for c in (0x04, 0x00, 0xFF):
        x = bytes([c])
        cases += [(x, x), (x * 3, x * 5), (b"ACGT" + x, x + b"ACGT" + x), (x + b"NNNN" + x * 2, b"NNNN" + x),
                  (bytes([c, 0x04, 0x00, 0xFF]), bytes([0xFF, 0x00, 0x04, c]) * 3), (x * 17, x * 16), (x * 16, x * 17)]
    cases.append((bytes(range(256)), bytes(range(255, -1, -1))))
    cases.append((bytes(range(256))[::3], bytes(range(256))))
    s1, s2 = [a for a, _ in cases], [b for _, b in cases]
    for p in (O.DEFAULT, (2, 0, 1, 1), (0, -1, 0, 0)):
        rows, _, err = emu(s1, s2, p)
        assert err == 0
        _check(rows, s1, s2, p)


def test_case_is_a_mismatch(emu):
    """Upper and lower case differ: 'acgt' against 'ACGT' scores 0, 'ACgT' against 'ACGT' is a mismatch in the middle."""
    s1 = [b"acgtacgt", b"ACgTACGTAC", b"nnnnACGT", b"ACGTNNNN"]
    s2 = [b"ACGTACGT", b"ACGTACGTAC", b"NNNNACGT", b"ACGTnnnn"]
    rows, _, err = emu(s1, s2, O.DEFAULT)
    assert err == 0
    _check(rows, s1, s2, O.DEFAULT)
    assert [r[1] for r in rows] == [0, 8, 4, 4]


def test_ties_swaps_empty_and_zero(emu):
    """Equally good alignments competing (a gap sliding along a run of N, neighbouring I and D), pairs the packer swaps,
    empty sequences and pairs that score 0."""
    cases = [
        (b"ACGTNNNNNNGTCA", b"ACGTNNNNGTCA", O.DEFAULT),
        (b"ACGTNNNNNNGTCA", b"ACGTNNNNGTCA", (2, -3, 5, 1)),
        (b"MKVLAAGGQQWW", b"MKVLGGQQWW", (2, -3, 5, 1)),
        (b"NNNNNNNNNN", b"NNNNN", (2, -1, 1, 3)),
        (b"RRRRYYRRRR", b"RRRRRRRR", (2, -1, 1, 3)),
        (b"ACGTTGCAACGT", b"ACGTGCAAACGT", (1, -3, 1, 1)),
        (b"CCGGTT", b"AANCCGGTTNAA", O.DEFAULT),
        (b"AANCCGGTTNAA", b"CCGGTT", O.DEFAULT),
        (b"", b"NNNN", O.DEFAULT),
        (b"N", b"", O.DEFAULT),
        (b"", b"", O.DEFAULT),
        (b"N", b"A", O.DEFAULT),
        (b"WWWW", b"YYYYYYYY", (3, -2, 2, 2)),
    ]
    for a, b, p in cases:
        rows, _, err = emu([a], [b], p)
        assert err == 0
        _check(rows, [a], [b], p)
    rows, _, _ = emu([b""], [b"NNNN"], O.DEFAULT)
    assert rows[0][:4] == (0, 0, (0, 0, 0, 0), 0)


def test_pool_and_pending_rounds(emu):
    """Slots too small for any rectangle and a pool with room for about one: pool pieces and later rounds, same results."""
    s1, s2 = _pairs(91, ALPHABETS["iupac"], 20, max_read=80, max_win=160)
    for p in (O.DEFAULT, (2, -3, 5, 1)):
        rows, rounds, err = emu(s1, s2, p, slot_words=4, pool_words=1)
        assert err == 0 and rounds > 1
        _check(rows, s1, s2, p)


def test_ops_stride_overflow(emu):
    """ops_count = -(operations) where ops_stride is too small, nothing written; the other pairs complete."""
    s1, s2 = _pairs(92, ALPHABETS["protein"], 12, max_read=80, max_win=140)
    p = (2, -3, 5, 1)
    rows, _, err = emu(s1, s2, p, ops_stride=3)
    assert err == 0
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align(a, b, p)
        _, score, span, n, runs = rows[k]
        assert (score, span) == (want[0], want[1])
        if len(want[2]) > 3:
            assert n == -len(want[2]) and runs == []
        else:
            assert n == len(want[2]) and runs == want[2]


@pytest.mark.parametrize("p", [O.DEFAULT, (2, -1, 1, 3), (5, -4, 11, 1)])
def test_acgt_bytes_equal_two_bit(emu, p):
    """On A,C,G,T input the byte bodies give exactly what the 2-bit bodies give: score, span, operations, counts."""
    r = np.random.default_rng(7)
    s1, s2 = [], []
    for k in range(40):
        w = rng.random_acgt(17, 2 * k, int(r.integers(1, 300)))
        rl = int(r.integers(0, 151))
        if k % 2 == 0 and len(w) > rl > 4:
            o = int(r.integers(0, len(w) - rl))
            rd = rng.mutate(w[o:o + rl], 17, 2 * k + 1, 0.06, 0.03)
        else:
            rd = rng.random_acgt(17, 2 * k + 1, rl)
        s1.append(bytes(rd)); s2.append(bytes(w))
        if k % 3 == 1:
            s1[-1], s2[-1] = s2[-1], s1[-1]
    by, r8, e8 = emu(s1, s2, p, bits=8, ops_stride=40)
    two, r2, e2 = emu(s1, s2, p, bits=2, ops_stride=40)
    assert e8 == e2 == 0 and r8 == r2
    assert by == two
    assert [row[1] for row in by] == O.gotoh_batch(s1, s2, p).tolist()
