"""swb200_align's blocked traceback (csrc/swb_traceback.cuh) without a GPU: tests/emu/align_blocks_emu.cu runs the product's
mode-10 direction kernel body, the checkpoint hand-over and the walk on CPU threads, once over the whole span and once in
blocks of rows (forward sweep with checkpoints, then recompute-and-walk from the bottom block up).  Every direction
nibble of the blocked launches must equal the one-launch nibble of the same cell, the two walks must write the same
operations, the score must be the oracle's, and the alignment must re-score to it over the whole span.  Needs nvcc (host
compile only)."""
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng
from test_align_batch_emu import PARAMS

EMU_DIR = Path(__file__).resolve().parent / "emu"

pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    work = tmp_path_factory.mktemp("align_blocks_emu")
    exe = work / "align_blocks_emu"
    subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe),
                    str(EMU_DIR / "align_blocks_emu.cu"), "-lpthread"], check=True, cwd=EMU_DIR)

    def run(a, b, p, block_rows, slack=1, warps=3):
        """a = seq1, b = seq2 (whole sequences); the driver gets the oracle's span.  Returns (span, parsed output)."""
        score, i0, j0, i1, j1 = O.gotoh_span(a, b, p)
        assert score > 0
        qf, tf = work / "q.bin", work / "t.bin"
        qf.write_bytes(bytes(b[i0 - 1:i1]))
        tf.write_bytes(bytes(a[j0 - 1:j1]))
        out = subprocess.run([str(exe), str(qf), str(tf), str(slack), str(warps), str(block_rows), *map(str, p)],
                             capture_output=True, text=True, timeout=900, check=True).stdout
        d = dict(kv.split("=", 1) for kv in out.split())
        d = {k: (v if k == "cigar" else int(v)) for k, v in d.items()}
        return score, (i0, j0, i1, j1), d
    return run


def rescore(cigar, a, b, span, p):
    """Walks the driver's M/I/D operations over seq1[j_start-1 ..] x seq2[i_start-1 ..]: (score, consumed the span,
    (first row, last row) of every gap run in span rows, as ('I' | 'D', rows before it, rows after it))."""
    ma, mi, gi, ge = p
    i0, j0, i1, j1 = span
    i, j, total, gaps = 0, 0, 0, []
    for cnt, op in re.findall(r"(\d+)([MID])", cigar):
        cnt = int(cnt)
        if op == "M":
            seg_a, seg_b = np.asarray(a[j0 - 1 + j:j0 - 1 + j + cnt]), np.asarray(b[i0 - 1 + i:i0 - 1 + i + cnt])
            assert len(seg_a) == cnt and len(seg_b) == cnt
            eq = int(np.count_nonzero(seg_a == seg_b))
            total += eq * ma + (cnt - eq) * mi
            i += cnt; j += cnt
        else:
            total -= gi + (cnt - 1) * min(gi, ge)       # gap_ext > gap_init: a run of k is k gaps of one (the walk merges them)
            gaps.append((op, i, i + (cnt if op == "D" else 0)))
            if op == "I":
                j += cnt
            else:
                i += cnt
    return total, (i, j) == (i1 - i0 + 1, j1 - j0 + 1), gaps


def check(emu, a, b, p, block_rows, slack=1, warps=3):
    score, span, d = emu(a, b, p, block_rows, slack, warps)
    rows = span[2] - span[0] + 1
    nb = -(-rows // 256)
    blocks = -(-nb // (block_rows // 256))
    assert (d["score"], d["blocked"], d["status"]) == (score, score, 0), (p, d, score)
    assert d["blocks"] == blocks and d["launches"] == 2 * blocks - 1, (d, rows)
    assert d["differing"] == 0, d                     # every recorded nibble is the one-launch nibble
    assert d["same_ops"] == 1, d                      # the blocked walk is the one-block walk
    total, whole, gaps = rescore(d["cigar"], a, b, span, p)
    assert whole and total == score, (p, total, score)
    return span, d, gaps


def planted(seed, n, sub, indel, flanks):
    a = rng.random_acgt(seed, 0, n)
    b = rng.mutate(a, seed, 1, sub, indel)
    if flanks:
        a = np.concatenate([rng.random_acgt(seed, 2, 90), a, rng.random_acgt(seed, 3, 40)])
        b = np.concatenate([rng.random_acgt(seed, 4, 33), b, rng.random_acgt(seed, 5, 120)])
    return a, b


@pytest.mark.parametrize("slack", [0, 1])
@pytest.mark.parametrize("k", range(len(PARAMS)))
def test_blocks_match_the_one_launch_traceback(emu, k, slack):
    """Planted pairs under the six parameter sets, span rows not a multiple of 256: blocks of 256 rows (three or more,
    two warps) and of 512 rows (a block of two bands on three warps)."""
    p = PARAMS[k]
    a, b = planted(1300 + k, 600 + 37 * k, 0.08, 0.04, k % 2 == 1)
    span, d, _ = check(emu, a, b, p, 256, slack, warps=2)
    rows = span[2] - span[0] + 1
    assert rows % 256 and d["blocks"] >= 3, rows
    check(emu, a, b, p, 512, slack, warps=3)


@pytest.mark.parametrize("slack", [0, 1])
def test_block_with_more_bands_than_warps(emu, slack):
    """A block of four bands on three warps: the band window of one launch goes round the ring of warps."""
    a, b = planted(1390, 1100, 0.06, 0.03, False)
    _, d, _ = check(emu, a, b, (2, -3, 5, 1), 1024, slack, warps=3)
    assert d["blocks"] == 2


@pytest.mark.parametrize("slack", [0, 1])
def test_block_edge_inside_a_vertical_gap(emu, slack):
    """30 extra bases of seq2 at rows 241-270: with affine costs one D run, and the edge at row 256 cuts it."""
    p = (2, -3, 5, 1)
    x = rng.random_acgt(1400, 0, 650)
    a, b = x, np.concatenate([x[:240], rng.random_acgt(1400, 1, 30), x[240:]])
    span, d, gaps = check(emu, a, b, p, 256, slack)
    assert span[:2] == (1, 1)
    assert any(op == "D" and before < 256 < after and after - before >= 25 for op, before, after in gaps), gaps


@pytest.mark.parametrize("row", [255, 256, 257])
def test_block_edge_next_to_a_horizontal_gap(emu, row):
    """25 extra bases of seq1 after row `row` of seq2: one I run at the block edge, just above or just below it."""
    p = (2, -3, 5, 1)
    x = rng.random_acgt(1410 + row, 0, 640)
    a, b = np.concatenate([x[:row], rng.random_acgt(1410 + row, 1, 25), x[row:]]), x
    span, d, gaps = check(emu, a, b, p, 256, 1)
    assert span[:2] == (1, 1)
    assert any(op == "I" and abs(before - row) <= 3 for op, before, _ in gaps), gaps   # the gap may slide over equal bases


def test_walk_crosses_a_block_edge_at_column_1(emu):
    """Free gaps: "AC" against A, 400 T, C aligns as 1=400D1=, so the walk meets the edges at rows 256 (and the
    recompute runs over one column)."""
    a, b = np.frombuffer(b"AC", np.uint8), np.frombuffer(b"A" + b"T" * 400 + b"C", np.uint8)
    span, d, _ = check(emu, a, b, (1, -1, 0, 0), 256, 1)
    assert span == (1, 1, 402, 2) and d["cigar"] == "1M400D1M" and d["edge_col"] == 1, (span, d)
