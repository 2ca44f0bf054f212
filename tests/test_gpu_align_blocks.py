"""swb200_align's blocked traceback: when the span's directions do not fit in device memory, pass 3 runs in blocks of rows
(forward sweep with one checkpoint row per block, then recompute-and-walk from the bottom block up).  Forced with
"align_block_rows", it must give byte for byte what the one-block traceback gives; on the 1 000 000 x 1 000 000 pair, whose
directions (about 500 GB) cannot fit, it runs by itself.  Engine launches tell which path ran: passes 1 and 2, B forward
launches, B - 1 recomputes."""
import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import api, rng
from concurrentproject_b200._lib import SwbError
from test_gpu_align import rescore

pytestmark = pytest.mark.gpu


@pytest.fixture
def block_rows():
    yield lambda v: api.configure("align_block_rows", v)
    api.configure("align_block_rows", 0)


def _blocks(span, k):
    bands = -(-(span[2] - span[0] + 1) // 256)
    return -(-bands // (k // 256))


def _cases():
    """The pairs of test_gpu_align.py: the six parameter sets, then the edge cases (ACGT only)."""
    cases = []
    for k, (n, sub, indel, p) in enumerate([(300, 0.06, 0.03, O.DEFAULT), (2000, 0.10, 0.05, (2, -3, 5, 1)), (5000, 0.08, 0.04, (5, -4, 11, 1)),
                                            (1500, 0.15, 0.08, (1, -1, 0, 0)), (3000, 0.05, 0.02, (3, -2, 2, 2)), (700, 0.3, 0.1, (2, -1, 3, 1))]):
        a = rng.random_acgt(800 + k, 0, n)
        b = rng.mutate(a, 800 + k, 1, sub, indel)
        if k % 2:
            a = np.concatenate([rng.random_acgt(800 + k, 2, 333), a, rng.random_acgt(800 + k, 3, 100)])
            b = np.concatenate([rng.random_acgt(800 + k, 4, 77), b, rng.random_acgt(800 + k, 5, 512)])
        cases.append((a, b, p))
    cases.append((np.frombuffer(b"ACGT" * 50, np.uint8), np.frombuffer(b"ACGT" * 50, np.uint8), O.DEFAULT))
    cases.append((np.frombuffer(b"TTTTACGTACGTTTTT", np.uint8), np.frombuffer(b"GGACGTACGTGG", np.uint8), O.DEFAULT))
    a = rng.random_acgt(850, 0, 4000)
    b = np.concatenate([a[:2000], a[2007:]])
    cases += [(a, b, (2, -3, 5, 1)), (a, b, O.DEFAULT)]
    return cases


def test_forced_blocks_give_the_one_block_alignment(block_rows):
    for a, b, p in _cases():
        block_rows(0)
        want = api.align(a, b, p)
        assert api.last_run()["engine_launches"] == 3
        for k in (256, 512):
            block_rows(k)
            got = api.align(a, b, p)
            assert got == want, (p, k, got[:2], want[:2])
            assert api.last_run()["engine_launches"] == 2 + 2 * _blocks(want[1], k) - 1, (p, k, want[1])


def test_forced_blocks_other_bytes_and_score_zero(block_rows):
    """Bytes other than A, C, G, T (byte-compare kernels) and pairs without an alignment give the same results in blocks."""
    pairs = [(b"HELLOWORLDGATTACAHELLO", b"XXWORLDGATTTACAYY"), (b"AAAA", b"CCCC"), (b"", b"ACGT"),
             (b"N" * 300 + b"ACGTACGTAC" * 40, b"ACGTACGTAC" * 40 + b"N" * 200)]
    for x, y in pairs:
        block_rows(0)
        want = api.align(x, y)
        block_rows(256)
        assert api.align(x, y) == want


def test_config2_pair_in_blocks(block_rows):
    """The 100 000 x 100 000 pair of BASELINE config 2 in blocks of 8 192 rows: the one-block CIGAR, byte for byte."""
    a, b = rng.random_acgt(2, 0, 100000), rng.random_acgt(2, 1, 100000)
    want = api.align(a, b)
    assert want[0] == 11446
    block_rows(8192)
    got = api.align(a, b)
    assert got == want
    nblocks = _blocks(want[1], 8192)
    assert nblocks >= 8 and api.last_run()["engine_launches"] == 2 + 2 * nblocks - 1


def test_n1m_pair_aligns_in_blocks():
    """1 000 000 x 1 000 000 (bench.py --workload n1m): the directions of its span cannot fit, so the library blocks by itself."""
    a, b = rng.random_acgt(6, 0, 1000000), rng.random_acgt(6, 1, 1000000)
    score, span, cigar = api.align(a, b)
    launches = api.last_run()["engine_launches"]
    assert score == 114366
    assert (score,) + span == api.score_span(a, b)
    assert rescore(cigar, a, b, span, O.DEFAULT) == (score, True)
    assert launches > 3


def test_align_block_rows_must_be_a_multiple_of_256(block_rows):
    for bad in (100, -256, 255, "x"):
        with pytest.raises(SwbError) as e:
            block_rows(bad)
        assert e.value.code == -2
