"""Batch alignment (csrc/swb_align_batch.cuh) without a GPU: the per-pair kernel bodies run on CPU threads
(tests/emu/align_batch_emu.cu, one pthread per lane of an emulated warp, the host driver's trace rounds) against a small
pure-Python reference of the contract -- end cell, start cell, directions over the span rectangle, walk -- that is itself
pinned to the C oracle's score and span on every case.  Needs nvcc (host compile only)."""
import ctypes as C
import re
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

EMU_DIR = Path(__file__).resolve().parent / "emu"
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")

PARAMS = [O.DEFAULT, (2, -3, 5, 1), (3, -2, 2, 2), (2, -1, 1, 3), (1, -1, 0, 0), (5, -4, 11, 1)]
NEG = -(1 << 29)
OPS = {1: "I", 2: "D", 7: "=", 8: "X"}


# ---- the reference ---------------------------------------------------------------------------------------------------
# seq1 = a (columns j), seq2 = b (rows i); E = a base of seq1 against a gap (along j), F = a base of seq2 against a gap.
def _track(h, i, j, best):
    b, bi, bj = best
    return (h, i, j) if h > b or (h == b and h > 0 and (j < bj or (j == bj and i < bi))) else best


def _local_end(a, b, p):
    ma, mi, gi, ge = p
    n = len(a)
    H, F = [0] * (n + 1), [0] * (n + 1)
    best = (0, 0, 0)
    for i in range(1, len(b) + 1):
        bc, e, hleft, hdiag = b[i - 1], 0, 0, 0
        for j in range(1, n + 1):
            e = max(e - ge, hleft - gi)
            f = max(F[j] - ge, H[j] - gi)
            h = max(hdiag + (ma if a[j - 1] == bc else mi), e, f, 0)
            hdiag, H[j], F[j], hleft = H[j], h, f, h
            best = _track(h, i, j, best)
    return best


def _anchored(a, b, p, dirs=False):
    """Every path starts at (0, 0); borders -(gi + (k-1) * min(gi, ge)).  Returns (max, i, j) or (H at the last cell, D)."""
    ma, mi, gi, ge = p
    gm, n = min(gi, ge), len(a)
    H = [0] + [-(gi + (j - 1) * gm) for j in range(1, n + 1)]
    F = [NEG] * (n + 1)
    D, best = [], (0, 0, 0)
    for i in range(1, len(b) + 1):
        bc, hdiag = b[i - 1], H[0]
        H[0] = -(gi + (i - 1) * gm)
        e, hleft, row = NEG, H[0], []
        for j in range(1, n + 1):
            e_ext, e_open, f_ext, f_open = e - ge, hleft - gi, F[j] - ge, H[j] - gi
            e, f = max(e_ext, e_open), max(f_ext, f_open)
            d = hdiag + (ma if a[j - 1] == bc else mi)
            h = max(d, e, f)
            if dirs:
                row.append((0 if h == d else (1 if h == e else 2)) | (4 if e_ext > e_open else 0) | (8 if f_ext > f_open else 0))
            hdiag, H[j], F[j], hleft = H[j], h, f, h
            best = _track(h, i, j, best)
        D.append(row)
    return (H[n], D) if dirs else best


def _walk(a, b, D, p):
    """From the last cell back to (0, 0): diagonal / E / F as the cell says; a gap that was opened ends its run when
    gap_ext > gap_init (two gaps, not one extended gap)."""
    split = p[3] > p[2]
    i, j, state, runs, brk = len(b), len(a), 0, [], False

    def emit(op, c):
        if runs and runs[-1][0] == op and not brk:
            runs[-1][1] += c
        else:
            runs.append([op, c])

    while i > 0 and j > 0:
        d = D[i - 1][j - 1]
        if state == 0:
            if d & 3 == 0:
                emit("=" if a[j - 1] == b[i - 1] else "X", 1); brk = False
                i, j = i - 1, j - 1
            else:
                state = d & 3
        elif state == 1:
            emit("I", 1)
            opened = not d & 4
            state, j, brk = (0 if opened else 1), j - 1, opened and split
        else:
            emit("D", 1)
            opened = not d & 8
            state, i, brk = (0 if opened else 2), i - 1, opened and split
    if j > 0:
        emit("I", j)
    if i > 0:
        emit("D", i)
    return [(op, c) for op, c in reversed(runs)]


def ref_align(a, b, p):
    """(score, (i_start, j_start, i_end, j_end), [(op, count), ...]) of the contract."""
    a, b = bytes(a), bytes(b)
    s, ie, je = _local_end(a, b, p)
    if s <= 0:
        return 0, (0, 0, 0, 0), []
    s2, ri, rj = _anchored(a[:je][::-1], b[:ie][::-1], p)
    assert s2 == s
    i0, j0 = ie - ri + 1, je - rj + 1
    ra, rb = a[j0 - 1:je], b[i0 - 1:ie]
    h, D = _anchored(ra, rb, p, dirs=True)
    assert h == s
    return s, (i0, j0, ie, je), _walk(ra, rb, D, p)


def rescore(runs, a, b, span, p):
    """main.cpp's costs over the span: MATCH / MISMATCH per pair, G_INIT + (k-1) G_EXT per gap operation of length k."""
    ma, mi, gi, ge = p
    i, j, total = span[0] - 1, span[1] - 1, 0
    for op, c in runs:
        if op in "=X":
            assert all((a[j + t] == b[i + t]) == (op == "=") for t in range(c))
            total += c * (ma if op == "=" else mi)
            i, j = i + c, j + c
        else:
            total -= gi + (c - 1) * ge
            if op == "I":
                j += c
            else:
                i += c
    assert (i, j) == (span[2], span[3])
    return total


# ---- the emulator ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    exe = EMU_DIR / "align_batch_emu"
    src = EMU_DIR / "align_batch_emu.cu"
    hdrs = [EMU_DIR.parent.parent / "concurrentproject_b200" / "csrc" / h for h in ("swb_align_batch.cuh", "swb_device.cuh")]
    if not exe.exists() or exe.stat().st_mtime < max(x.stat().st_mtime for x in [src] + hdrs):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(src),
                        "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("align_batch_emu")

    def run(s1, s2, p, slot_words=4096, pool_words=0, ops_stride=None):
        if ops_stride is None:
            ops_stride = max(1, max(len(a) + len(b) for a, b in zip(s1, s2)))
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(exe), str(f), *map(str, [*p, slot_words, pool_words, ops_stride])], capture_output=True,
                             text=True, timeout=900, check=True).stdout.strip().split("\n")
        rows = []
        for line in res[:-1]:
            v = [int(x) for x in line.split()]
            rows.append((v[0], tuple(v[1:5]), v[5], [(OPS[w & 15], w >> 4) for w in v[6:]]))
        rounds, err = re.fullmatch(r"rounds (\d+) err (\d+)", res[-1]).groups()
        return rows, int(rounds), int(err)
    return run


def _pairs(seed, npairs, max_read=150, max_win=400):
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(npairs):
        w = rng.random_acgt(seed, 2 * k, int(r.integers(1, max_win + 1)))
        rl = int(r.integers(0, max_read + 1))
        if k % 2 == 0 and len(w) > rl > 4:
            o = int(r.integers(0, len(w) - rl))
            rd = rng.mutate(w[o:o + rl], seed, 2 * k + 1, 0.06, 0.03)
        else:
            rd = rng.random_acgt(seed, 2 * k + 1, rl)
        if k % 3 == 1:
            s1.append(bytes(w)); s2.append(bytes(rd))        # the read as seq2 as well: both orientations of the packer
        else:
            s1.append(bytes(rd)); s2.append(bytes(w))
    return s1, s2


def _check(rows, s1, s2, p):
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align(a, b, p)
        assert (want[0],) + want[1] == O.gotoh_span(a, b, p), (k, p)            # the reference is the oracle's score and span
        score, span, n, runs = rows[k]
        assert (score, span, runs) == want, (k, p, score, span, runs[:8], want[0], want[1], want[2][:8])
        assert n == len(runs)
        if score > 0:
            assert rescore(runs, a, b, span, p) == score, (k, p)


@pytest.mark.parametrize("p", PARAMS)
def test_align_batch_kernel_bodies(emu, p):
    """37 ragged pairs (reads 0..150, windows 1..400, planted and random, both orientations): two passes of the warp, the
    second one partly empty."""
    s1, s2 = _pairs(70 + PARAMS.index(p), 37)
    rows, rounds, err = emu(s1, s2, p)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, p)


def test_pool_and_pending_rounds(emu):
    """Slots too small for any rectangle and a pool with room for about one: every pair takes a piece of the pool or waits
    for a later round, and the results do not change."""
    s1, s2 = _pairs(91, 20, max_read=120, max_win=200)
    for p in (O.DEFAULT, (2, -3, 5, 1)):
        rows, rounds, err = emu(s1, s2, p, slot_words=4, pool_words=1)
        assert err == 0 and rounds > 1
        _check(rows, s1, s2, p)


def test_ops_stride_overflow(emu):
    """ops_count = -(operations) where ops_stride is too small, nothing written; the other pairs complete."""
    s1, s2 = _pairs(92, 12, max_read=100, max_win=160)
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


def test_tie_rules(emu):
    """Where equally good alignments compete: a gap sliding along a run of equal bases, one long deletion under affine
    gaps, neighbouring I and D, alignments that touch row 0 / column 0 of the span, and pairs the packer swaps."""
    cases = [
        (b"ACGTAAAAAAGTCA", b"ACGTAAAAGTCA", O.DEFAULT),
        (b"ACGTAAAAAAGTCA", b"ACGTAAAAGTCA", (2, -3, 5, 1)),
        (b"GGGGCCCCAAAATTTT", b"GGGGAAAATTTT", (2, -3, 5, 1)),
        (b"ACGTTGCAACGT", b"ACGTGCAAACGT", (1, -3, 1, 1)),
        (b"ACGTACGTTACGTACGT", b"ACGTACGTCACGTACGT", (1, -3, 1, 1)),
        (b"AACCGGTTAACC", b"CCGGTT", O.DEFAULT),
        (b"CCGGTT", b"AACCGGTTAACC", O.DEFAULT),
        (b"TTTTTTTTTT", b"TTTTT", (2, -1, 1, 3)),
        (b"AAAACCAAAA", b"AAAAAAAA", (2, -1, 1, 3)),
        (b"ACGATCGATCGTAGCTAGCTAGCT", b"ACGATCGTCGTAGCTTAGCTAGCT", (1, -1, 0, 0)),
        (b"A", b"A", O.DEFAULT),
        (b"A", b"C", O.DEFAULT),
        (b"", b"ACGT", O.DEFAULT),
    ]
    x = rng.random_acgt(5, 0, 300)
    cases.append((bytes(x), bytes(np.concatenate([x[:140], x[147:]])), (2, -3, 5, 1)))
    cases.append((bytes(np.concatenate([x[:100], x[103:200]])), bytes(x[:200]), (5, -4, 11, 1)))
    for a, b, p in cases:
        rows, _, err = emu([a], [b], p)
        assert err == 0
        _check(rows, [a], [b], p)
    # a split gap under gap_ext > gap_init: two neighbouring gap characters are two opened gaps
    s, span, runs = ref_align(b"AAAACCAAAA", b"AAAAAAAA", (2, -1, 1, 3))
    assert s == 14 and [op for op, _ in runs].count("I") == 2 and ("I", 2) not in runs


# ---- the C ABI refuses bad arguments before it touches a device ------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def test_align_batch_argument_errors_need_no_gpu(lib):
    from concurrentproject_b200 import _lib
    LL, I, U = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_uint)

    def call(s1, s2, p=(1, -1, 1, 1), stride=8, l1=None, null_out=False):
        f1, f2 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy(), np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
        len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
        len2 = np.array([len(x) for x in s2], np.int32)
        o1 = np.concatenate([[0], np.cumsum([len(x) for x in s1])[:-1]]).astype(np.int64)
        o2 = np.concatenate([[0], np.cumsum([len(x) for x in s2])[:-1]]).astype(np.int64)
        n = len(s1)
        sc, sp, ops, cnt = np.zeros(n, np.int32), np.zeros(4 * n, np.int32), np.zeros(n * stride + 1, np.uint32), np.zeros(n, np.int32)
        pp = _lib.Params(*p)
        return lib.swb200_align_batch(f1.ctypes.data_as(C.POINTER(C.c_ubyte)), o1.ctypes.data_as(LL), len1.ctypes.data_as(I),
                                      f2.ctypes.data_as(C.POINTER(C.c_ubyte)), o2.ctypes.data_as(LL), len2.ctypes.data_as(I), n,
                                      C.byref(pp), None, sc.ctypes.data_as(I), None if null_out else sp.ctypes.data_as(I),
                                      ops.ctypes.data_as(U), stride, cnt.ctypes.data_as(I))

    ok = ([b"ACGT"], [b"ACGTT"])
    assert call(*ok, null_out=True) == -2                                        # null output
    assert call(*ok, stride=0) == -2 and b"argument" in lib.swb200_last_error()  # ops_stride < 1
    assert call(*ok, l1=[-1]) == -2                                              # negative length
    assert call(*ok, p=(1, 1, 1, 1)) == -2 and b"limits" in lib.swb200_last_error()
    assert call([b"A" * 1025], [b"C" * 1100]) == -2 and b"1024" in lib.swb200_last_error()
    assert call([b"A" * 700], [b"C" * 800], p=(50, -1, 1, 1)) == -6                # match * min(len) > 32766 - match
    assert lib.swb200_align_batch(None, None, None, None, None, None, 0, None, None, None, None, None, 1, None) == 0
    assert lib.swb200_align_batch(None, None, None, None, None, None, -1, None, None, None, None, None, 1, None) == -2
    assert lib.swb200_batch_align(None, None, None, None, None, None, None, 8, None) == -2
