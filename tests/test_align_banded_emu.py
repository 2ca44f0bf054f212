"""Banded batch alignment (csrc/swb_align_banded.cuh) without a GPU: the per-pair warp bodies run on CPU threads
(tests/emu/align_banded_emu.cu, one pthread per lane of two emulated warps, the host driver's trace rounds) against a
pure-Python reference of the contract -- banded local end cell, start cell by the anchored recurrence in the mirrored
band, banded directions over the span, walk -- that is itself pinned to the C checker (banded_oracle) and, where the
band covers the whole pair, to the unbanded reference of the read-batch tests.  Also: the C ABI of both banded
alignment calls refuses bad arguments before it touches a device.  Needs nvcc (host compile only)."""
import ctypes as C
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
from test_align_batch_emu import PARAMS, _track, _walk, ref_align, rescore

EMU_DIR = Path(__file__).resolve().parent / "emu"
NEG = -(1 << 29)
OPS = {1: "I", 2: "D", 7: "=", 8: "X"}
needs_nvcc = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


# ---- the reference ---------------------------------------------------------------------------------------------------
# seq1 = a (columns j), seq2 = b (rows i); cell (i, j) is in the band iff lo <= j - i <= hi.
def _banded_local_end(a, b, p, lo, hi):
    """main.cpp:57-63 on in-band cells; out-of-band cells are H = E = F = 0 (oracle_gotoh_banded).  (score, i, j)."""
    ma, mi, gi, ge = p
    n, m = len(a), len(b)
    H = [[0] * (n + 1) for _ in range(m + 1)]
    E = [[0] * (n + 1) for _ in range(m + 1)]
    F = [[0] * (n + 1) for _ in range(m + 1)]
    best = (0, 0, 0)
    for i in range(1, m + 1):
        for j in range(max(1, i + lo), min(n, i + hi) + 1):
            E[i][j] = max(E[i][j - 1] - ge, H[i][j - 1] - gi)
            F[i][j] = max(F[i - 1][j] - ge, H[i - 1][j] - gi)
            H[i][j] = max(H[i - 1][j - 1] + (ma if a[j - 1] == b[i - 1] else mi), E[i][j], F[i][j], 0)
            best = _track(H[i][j], i, j, best)
    return best


def _banded_anchored(a, b, p, lo, hi, dirs=False):
    """The anchored recurrence from (0, 0) (lo <= 0 <= hi), cells outside the band unreachable; borders
    -(gi + (k-1) min(gi, ge)) where they are in the band.  (max, i, j), or (H at the last cell, directions)."""
    ma, mi, gi, ge = p
    gm, n, m = min(gi, ge), len(a), len(b)
    H = [[NEG] * (n + 1) for _ in range(m + 1)]
    E = [[NEG] * (n + 1) for _ in range(m + 1)]
    F = [[NEG] * (n + 1) for _ in range(m + 1)]
    for j in range(0, min(n, hi) + 1):
        H[0][j] = 0 if j == 0 else -(gi + (j - 1) * gm)
    for i in range(1, min(m, -lo) + 1):
        H[i][0] = -(gi + (i - 1) * gm)
    D = [[0] * n for _ in range(m)]
    best = (0, 0, 0)
    for i in range(1, m + 1):
        for j in range(max(1, i + lo), min(n, i + hi) + 1):
            e_ext, e_open = E[i][j - 1] - ge, H[i][j - 1] - gi
            f_ext, f_open = F[i - 1][j] - ge, H[i - 1][j] - gi
            e, f = max(e_ext, e_open), max(f_ext, f_open)
            d = H[i - 1][j - 1] + (ma if a[j - 1] == b[i - 1] else mi)
            h = max(d, e, f)
            D[i - 1][j - 1] = (0 if h == d else (1 if h == e else 2)) | (4 if e_ext > e_open else 0) | (8 if f_ext > f_open else 0)
            H[i][j], E[i][j], F[i][j] = h, e, f
            best = _track(h, i, j, best)
    return (H[m][n], D) if dirs else best


def ref_align_banded(a, b, p, lo, hi):
    """(score, (i_start, j_start, i_end, j_end), [(op, count), ...]) of the banded contract."""
    a, b = bytes(a), bytes(b)
    s, ie, je = _banded_local_end(a, b, p, lo, hi)
    if s <= 0:
        return 0, (0, 0, 0, 0), []
    s2, ri, rj = _banded_anchored(a[:je][::-1], b[:ie][::-1], p, (je - ie) - hi, (je - ie) - lo)
    assert s2 == s
    i0, j0 = ie - ri + 1, je - rj + 1
    ra, rb = a[j0 - 1:je], b[i0 - 1:ie]
    h, D = _banded_anchored(ra, rb, p, lo - (j0 - i0), hi - (j0 - i0), dirs=True)
    assert h == s
    return s, (i0, j0, ie, je), _walk(ra, rb, D, p)


def path_in_band(runs, span, lo, hi):
    """Every cell the alignment visits (aligned pairs and gap positions) lies in lo <= j - i <= hi."""
    i, j = span[0], span[1]
    cells = []
    for op, c in runs:
        for _ in range(c):
            cells.append((i, j))
            if op in "=X":
                i, j = i + 1, j + 1
            elif op == "I":
                j += 1
            else:
                i += 1
    return all(lo <= jj - ii <= hi for ii, jj in cells)


# ---- the reference against the C checker, without the emulator ------------------------------------------------------
def _pairs(seed, npairs, max_len=90, shift=0):
    """Ragged pairs: related (seq2 a mutated copy of seq1 shifted by `shift` bases) and unrelated, both directions."""
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(npairs):
        n = int(r.integers(0, max_len + 1))
        a = rng.random_acgt(seed, 2 * k, n + abs(shift))
        if k % 3 != 2:
            b = rng.mutate(a, seed, 2 * k + 1, 0.08, 0.04)
            a, b = (a[shift:], b) if shift >= 0 else (a, b[-shift:])
            b = b[:int(r.integers(0, max_len + 1))]
        else:
            a, b = a[:n], rng.random_acgt(seed, 2 * k + 1, int(r.integers(0, max_len + 1)))
        if k % 4 == 1:
            a, b = b, a
        s1.append(bytes(a)); s2.append(bytes(b))
    return s1, s2


BANDS = [(-32, 31), (5, 68), (-70, -7), (3, 66), (-66, -3), (-20, 43), (150, 213)]


@pytest.mark.parametrize("p", PARAMS)
def test_reference_is_pinned_to_the_oracle(p):
    s1, s2 = _pairs(30 + PARAMS.index(p), 14, max_len=70)
    for lo, hi in BANDS:
        for a, b in zip(s1, s2):
            want = ref_align_banded(a, b, p, lo, hi)
            assert want[0] == O.gotoh_banded(a, b, lo, hi, p)
            assert (want[0],) + want[1] == BO.gotoh_banded_span(a, b, lo, hi, p), (lo, hi, a, b)
            if want[0] > 0:
                assert rescore(want[2], a, b, want[1], p) == want[0]
                assert path_in_band(want[2], want[1], lo, hi)


@pytest.mark.parametrize("p", PARAMS)
def test_full_band_equals_the_unbanded_contract(p):
    """A band that covers the whole pair (band_lo <= -(len2-1), band_hi >= len1-1) gives the read-batch result."""
    s1, s2 = _pairs(40 + PARAMS.index(p), 16, max_len=30)
    for a, b in zip(s1, s2):
        for lo in sorted({-max(len(b) - 1, 0), -32, -63 + max(len(a) - 1, 0)}):
            hi = lo + 63
            if lo > -max(len(b) - 1, 0) or hi < len(a) - 1:
                continue
            assert ref_align_banded(a, b, p, lo, hi) == ref_align(a, b, p), (a, b, lo)
            assert BO.gotoh_banded_span(a, b, lo, hi, p) == O.gotoh_span(a, b, p)


def test_oracle_on_long_pairs():
    """The C checker on cfg5-like pairs: its score is oracle_gotoh_banded's, and its span stays in the band."""
    for k in range(3):
        a, b = rng.long_pair(5, k, 3000)
        for lo in (-32, -10, 2):
            s, i0, j0, i1, j1 = BO.gotoh_banded_span(a, b, lo, lo + 63)
            assert s == O.gotoh_banded(a, b, lo, lo + 63) > 0
            assert lo <= j0 - i0 <= lo + 63 and lo <= j1 - i1 <= lo + 63 and 1 <= i0 <= i1 and 1 <= j0 <= j1


# ---- the emulator ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    work = tmp_path_factory.mktemp("align_banded_emu")
    exe = work / "align_banded_emu"
    subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe),
                    str(EMU_DIR / "align_banded_emu.cu"), "-lpthread"], check=True)

    def run(s1, s2, p, lo, slot_words=1 << 16, pool_words=0, ops_stride=None):
        if ops_stride is None:
            ops_stride = max(1, max(len(a) + len(b) for a, b in zip(s1, s2)))
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(exe), str(f), *map(str, [lo, *p, slot_words, pool_words, ops_stride])], capture_output=True,
                             text=True, timeout=900, check=True).stdout.strip().split("\n")
        rows = []
        for line in res[:-1]:
            v = [int(x) for x in line.split()]
            rows.append((v[0], tuple(v[1:5]), v[5], [(OPS[w & 15], w >> 4) for w in v[6:]]))
        rounds, err = re.fullmatch(r"rounds (\d+) err (\d+) cells \d+", res[-1]).groups()
        return rows, int(rounds), int(err)
    return run


def _check(rows, s1, s2, p, lo, hi):
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align_banded(a, b, p, lo, hi)
        score, span, n, runs = rows[k]
        assert (score, span, runs) == want, (k, p, lo, score, span, runs[:8], want[0], want[1], want[2][:8])
        assert n == len(runs)
        if score > 0:
            assert rescore(runs, a, b, span, p) == score and path_in_band(runs, span, lo, hi), (k, p, lo)


@needs_nvcc
@pytest.mark.parametrize("p", PARAMS)
def test_align_banded_kernel_bodies(emu, p):
    """Ragged pairs (0..90 bases, related and unrelated, both orientations) under a centred band, and shifted pairs under
    bands wholly above and wholly below the main diagonal."""
    s1, s2 = _pairs(70 + PARAMS.index(p), 12)
    rows, rounds, err = emu(s1, s2, p, -32)
    assert err == 0 and rounds == 1
    _check(rows, s1, s2, p, -32, 31)
    for shift, lo in ((40, 20), (-40, -90)):
        s1, s2 = _pairs(80 + PARAMS.index(p), 6, max_len=120, shift=shift)
        rows, _, err = emu(s1, s2, p, lo)
        assert err == 0
        _check(rows, s1, s2, p, lo, lo + 63)


@needs_nvcc
def test_band_edges(emu):
    """Bands that exclude the unbanded optimum, cut row 1 / column 1, hold no cell of the pair, pairs shorter than the
    band, empty sequences, and runs of equal bases along the band's edge (ties between gap placements)."""
    x = rng.random_acgt(9, 0, 160)
    planted = bytes(x[70:150])                      # the unbanded optimum lies on diagonal j - i = -70 ...
    noise = bytes(rng.random_acgt(9, 1, 80))
    cases = [
        ([bytes(x[:10]) + planted], [noise + planted + noise[:20]], (2, -3, 5, 1), -32),   # ... band -32..31 misses it
        ([b"ACGTACGTAC" * 6], [b"ACGTACGTAC" * 6], O.DEFAULT, 3),       # cuts row 1 (j >= 4)
        ([b"ACGTACGTAC" * 6], [b"ACGTACGTAC" * 6], O.DEFAULT, -66),     # cuts column 1 (i >= 4)
        ([b"ACGT" * 5], [b"ACGT" * 5], O.DEFAULT, 40),                  # no cell of the pair in the band
        ([b"ACGT" * 5], [b"ACGT" * 5], O.DEFAULT, -90),
        ([b"ACGGT"], [b"ACGT"], (2, -3, 5, 1), -32),                     # shorter than the band
        ([b""], [b"ACGT"], O.DEFAULT, -32),
        ([b"ACGT"], [b""], O.DEFAULT, -32),
        ([b"A" * 40 + b"C" * 30], [b"A" * 70 + b"C" * 30], O.DEFAULT, -63),        # the gap slides to the band's edge
        ([b"A" * 70 + b"C" * 30], [b"A" * 40 + b"C" * 30], (2, -1, 1, 3), 0),
        ([b"TTTT" + b"G" * 50], [b"G" * 80], (1, -1, 0, 0), -31),
        ([b"AAAACCAAAA" * 4], [b"AAAAAAAA" * 4], (2, -1, 1, 3), -5),
    ]
    for s1, s2, p, lo in cases:
        rows, _, err = emu(s1, s2, p, lo)
        assert err == 0
        _check(rows, s1, s2, p, lo, lo + 63)
    assert ref_align_banded(cases[0][0][0], cases[0][1][0], (2, -3, 5, 1), -32, 31)[0] < O.gotoh_full(cases[0][0][0], cases[0][1][0], (2, -3, 5, 1))
    assert ref_align_banded(b"ACGT" * 5, b"ACGT" * 5, O.DEFAULT, 40, 103) == (0, (0, 0, 0, 0), [])


@needs_nvcc
def test_pool_and_pending_rounds(emu):
    """Slots too small for any span and a pool with room for about one: every pair takes a piece of the pool or waits
    for a later round, and the results do not change."""
    s1, s2 = _pairs(91, 10, max_len=80)
    for p in (O.DEFAULT, (2, -3, 5, 1)):
        rows, rounds, err = emu(s1, s2, p, -32, slot_words=4, pool_words=1)
        assert err == 0 and rounds > 1
        _check(rows, s1, s2, p, -32, 31)


@needs_nvcc
def test_ops_stride_overflow(emu):
    """ops_count = -(operations) where ops_stride is too small, nothing written; the other pairs complete."""
    s1, s2 = _pairs(92, 10, max_len=80)
    p = (2, -3, 5, 1)
    rows, _, err = emu(s1, s2, p, -32, ops_stride=3)
    assert err == 0
    for k, (a, b) in enumerate(zip(s1, s2)):
        want = ref_align_banded(a, b, p, -32, 31)
        score, span, n, runs = rows[k]
        assert (score, span) == (want[0], want[1])
        if len(want[2]) > 3:
            assert n == -len(want[2]) and runs == []
        else:
            assert n == len(want[2]) and runs == want[2]


# ---- the C ABI refuses bad arguments before it touches a device ------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from concurrentproject_b200 import _lib
    _lib.build()
    return _lib.load()


def test_align_banded_argument_errors_need_no_gpu(lib):
    from concurrentproject_b200 import _lib
    LL, I, U = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_uint)

    def call(s1, s2, lo=-32, hi=31, p=(1, -1, 1, 1), stride=8, l1=None, null_out=False):
        f1, f2 = np.frombuffer(b"".join(s1) or b"A", np.uint8).copy(), np.frombuffer(b"".join(s2) or b"A", np.uint8).copy()
        len1 = np.array(l1 if l1 is not None else [len(x) for x in s1], np.int32)
        len2 = np.array([len(x) for x in s2], np.int32)
        o1 = np.concatenate([[0], np.cumsum([len(x) for x in s1])[:-1]]).astype(np.int64)
        o2 = np.concatenate([[0], np.cumsum([len(x) for x in s2])[:-1]]).astype(np.int64)
        n = len(s1)
        sc, sp, ops, cnt = np.zeros(n, np.int32), np.zeros(4 * n, np.int32), np.zeros(n * stride + 1, np.uint32), np.zeros(n, np.int32)
        pp = _lib.Params(*p)
        return lib.swb200_align_banded_batch(f1.ctypes.data_as(C.POINTER(C.c_ubyte)), o1.ctypes.data_as(LL), len1.ctypes.data_as(I),
                                             f2.ctypes.data_as(C.POINTER(C.c_ubyte)), o2.ctypes.data_as(LL), len2.ctypes.data_as(I),
                                             n, lo, hi, C.byref(pp), None, sc.ctypes.data_as(I),
                                             None if null_out else sp.ctypes.data_as(I), ops.ctypes.data_as(U), stride,
                                             cnt.ctypes.data_as(I))

    ok = ([b"ACGT"], [b"ACGTT"])
    assert call(*ok, null_out=True) == -2                                        # null output
    assert call(*ok, stride=0) == -2 and b"argument" in lib.swb200_last_error()  # ops_stride < 1
    assert call(*ok, l1=[-1]) == -2                                              # negative length
    assert call(*ok, p=(1, 1, 1, 1)) == -2 and b"limits" in lib.swb200_last_error()
    assert call(*ok, p=(1, -1, 101, 1)) == -2
    assert call(*ok, lo=-32, hi=32) == -2 and b"64" in lib.swb200_last_error()  # band width != 64
    assert call(*ok, lo=0, hi=0) == -2
    assert call([b"A" * 700], [b"C" * 800], p=(50, -1, 1, 1)) == -6             # match * min(len) > 32766 - match
    assert lib.swb200_align_banded_batch(None, None, None, None, None, None, 0, -32, 31, None, None, None, None, None, 1, None) == 0
    assert lib.swb200_align_banded_batch(None, None, None, None, None, None, -1, -32, 31, None, None, None, None, None, 1, None) == -2
    assert lib.swb200_align_banded_batch(None, None, None, None, None, None, 0, -32, 40, None, None, None, None, None, 1, None) == -2
    assert lib.swb200_batch_align_banded(None, -32, 31, None, None, None, None, None, None, 8, None) == -2
