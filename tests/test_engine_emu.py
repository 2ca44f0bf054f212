"""Runs the product's wavefront engine body on CPU threads (tests/emu/engine_emu.cu) and compares
with the oracle.  This is how the hand-off protocol (tags, ring laps, back-pressure, ring
wrap-around over several rounds, multi-GPU ring) is covered without a GPU; the same source is what
the sm_100a kernels compile.  Needs nvcc (host compile only)."""
import os
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

EMU_DIR = Path(__file__).resolve().parent / "emu"
EMU = EMU_DIR / "engine_emu"

pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    src = EMU_DIR / "engine_emu.cu"
    hdrs = list((EMU_DIR.parent.parent / "concurrentproject_b200" / "csrc").glob("swb_*.cuh"))
    if not EMU.exists() or EMU.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(EMU),
                        str(src), "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("engine_emu")      # per run: concurrent runs and other users do not collide

    def run(q, t, R, mode, slack, W, G, p=O.DEFAULT, link_len=4096, epoch=5, tmp=work, final_row=False, short=None, hs=False):
        qf, tf, ff = tmp / "swb_emu_q.bin", tmp / "swb_emu_t.bin", tmp / "swb_emu_final.bin"
        qf.write_bytes(bytes(q)); tf.write_bytes(bytes(t))
        ma, mi, gi, ge = p
        env = dict(os.environ, EMU_FINAL=str(ff)) if final_row else dict(os.environ)
        env.pop("EMU_FINAL", None) if not final_row else None
        env.pop("EMU_SHORT", None)
        env.pop("EMU_HS", None)
        if hs:                                      # launch config 4: slack inside a thread as well
            env["EMU_HS"] = "1"
        if short is not None:                       # row-loop flavour; default: short chain iff slack == 1
            env["EMU_SHORT"] = str(int(short))
        out = subprocess.run([str(EMU), str(qf), str(tf), *map(str, [R, mode, slack, W, G, epoch, ma, mi, gi, ge, link_len])],
                             capture_output=True, text=True, timeout=900, check=True, env=env).stdout
        d = dict(kv.split("=") for kv in out.split())
        if mode in (6, 8): # end-cell tracking: (score, status, 1-based row in Q, 1-based position in T)
            return int(d["score"]), int(d["status"]), int(d["endrow"]) + 1, int(d["endpos"]) + 1, int(d["endh"])
        if not final_row:
            return int(d["score"]), int(d["status"])
        raw = ff.read_bytes()
        LT, skew = (int(x) for x in np.frombuffer(raw[:16], dtype=np.int64))
        ent = np.frombuffer(raw[16:], dtype=np.uint32).reshape(-1, 2)[:, 0][skew:skew + LT]
        lo = (ent & 0xFFFF).astype(np.int16).astype(np.int32)
        hi = (ent >> 16).astype(np.int16).astype(np.int32)
        return int(d["score"]), int(d["status"]), lo, hi
    return run


def planted(seed, n, sub=0.06, indel=0.03):
    a = rng.random_acgt(seed, 0, n)
    return a, rng.mutate(a, seed, 1, sub, indel)


@pytest.mark.parametrize("mode,slack", [(0, 1), (0, 0), (2, 1), (2, 0)])
def test_affine_engine_small(emu, mode, slack):
    cases = [(300, 1, 2, 1, O.DEFAULT), (700, 2, 3, 1, (2, -3, 5, 1)), (900, 3, 2, 2, (5, -4, 11, 1)),
             (450, 1, 1, 1, (2, -1, 3, 1)), (1200, 4, 2, 1, (1, -1, 4, 2))]
    if mode == 2:      # 32-bit lanes: bands are half as tall, the emulation twice as slow -- smaller cases, same shapes
        cases = [(200, 1, 2, 1, O.DEFAULT), (400, 2, 3, 1, (2, -3, 5, 1)), (500, 3, 2, 2, (5, -4, 11, 1)), (300, 1, 1, 1, (2, -1, 3, 1))]
    for k, (n, R, W, G, p) in enumerate(cases):
        a, b = planted(100 + k, n)
        assert emu(a, b, R, mode, slack, W, G, p) == (O.gotoh_rolling(a, b, p), 0), (n, R, W, G, p)
        if k % 2 == 0:
            assert emu(b, a, R, mode, slack, W, G, p) == (O.gotoh_rolling(a, b, p), 0)


@pytest.mark.parametrize("slack", [0, 1])
def test_linear_engine_small(emu, slack):
    for k, (n, R, W, G, p) in enumerate([(300, 1, 2, 1, O.DEFAULT), (800, 2, 3, 2, (3, -2, 2, 2)), (1000, 8, 1, 1, (1, -3, 1, 1))]):
        a, b = planted(200 + k, n)
        assert emu(a, b, R, 1, slack, W, G, p) == (O.gotoh_rolling(a, b, p), 0)


@pytest.mark.parametrize("short", [0, 1])
def test_row_loop_flavours_and_gap_open_cheaper_than_extension(emu, short):
    """Both row-loop flavours (swb_engine.cuh: SHORT = one dependent instruction per row, used by launch configs
    1 and 3; long = fewest instructions, config 2) under both slacks, including gap_init < gap_ext, where the short
    flavour carries F down a lane with -min(gap_ext, gap_init)."""
    a, b = planted(500, 300, 0.08, 0.05)
    for p in [(2, -1, 1, 3), (3, -2, 0, 0), (2, -3, 5, 1)]:
        want = O.gotoh_rolling(a, b, p)
        for mode, slack in ((0, 0), (0, 1), (2, 1 - short), (3, short)):
            assert emu(a, b, 2, mode, slack, 2, 1, p, short=short) == (want, 0), (p, mode, slack)
        if p[2] == p[3]:
            for mode in (1, 4):
                assert emu(b, a, 1, mode, short, 2, 1, p, short=short) == (want, 0), (p, mode)


@pytest.mark.parametrize("slack", [0, 1])
def test_end_cell_tracking(emu, slack):
    """32-bit tracking engine (SURVEY.md 8(f) row 4): the end cell of the best local alignment -- highest H, then the
    smallest T position, then the smallest Q row -- across lanes, bands, rounds and 128-step key windows; with zero
    gap costs (3,-2,0,0) whole plateaus of cells tie with the maximum."""
    for k, (nq, nt, R, W, p) in enumerate([(200, 700, 1, 2, O.DEFAULT), (300, 300, 2, 3, (3, -2, 0, 0)), (150, 900, 1, 1, (2, -3, 5, 1)),
                                           (260, 500, 4, 2, (1, -1, 0, 0))]):
        q = rng.random_acgt(900 + k, 0, nq)
        t = rng.random_acgt(900 + k, 1, nt)
        t[nt // 2: nt // 2 + 60] = q[20:80]                     # one planted common stretch ...
        if k % 2:
            t[nt // 4: nt // 4 + 60] = q[20:80]                 # ... or two equally good ones
        want, wi, wj = O.gotoh_end(t, q, p)                      # seq1 = T (columns j), seq2 = Q (rows i)
        score, status, row, pos, endh = emu(q, t, R, 6, slack, W, 1, p)
        assert (score, status, endh) == (want, 0, want)
        assert (row, pos) == (wi, wj), (k, nq, nt, R, W, p)


@pytest.mark.parametrize("slack", [0, 1])
def test_anchored_recurrence_finds_the_start_cell(emu, slack):
    """ANCH variant of the 32-bit engine: alignments start at the origin, no clamp at 0, gap-cost borders; the
    maximum and its position against the oracle's anchored DP, over several bands and rounds."""
    for k, (nq, nt, R, W, p) in enumerate([(150, 200, 1, 2, O.DEFAULT), (300, 260, 2, 3, (3, -2, 4, 1)), (200, 330, 1, 1, (2, -3, 1, 3)),
                                           (260, 120, 4, 2, (1, -1, 0, 0))]):
        core = rng.random_acgt(950 + k, 0, min(nq, nt) // 2)
        q = np.concatenate([rng.mutate(core, 950 + k, 5, 0.06, 0.03), rng.random_acgt(950 + k, 1, nq)])[:nq]
        t = np.concatenate([core, rng.random_acgt(950 + k, 2, nt)])[:nt]
        want, wi, wj = O.gotoh_anchored_end(t, q, p)             # seq1 = T (columns j), seq2 = Q (rows i)
        assert want > 0
        score, status, row, pos, endh = emu(q, t, R, 8, slack, W, 1, p)
        assert (status, endh) == (0, want), (k, p)
        assert (row, pos) == (wi, wj), (k, nq, nt, R, W, p)


def test_edge_shapes(emu):
    for q, t in [(b"A", b"A"), (b"A", b"G"), (b"ACGT" * 16, b"A"), (b"A", b"ACGT" * 16), (b"A" * 129, b"A" * 129),
                 (b"A" * 200, b"T" * 200), (b"ACGT" * 50, b"GCTA" * 50 + b"G")]:
        for mode in (0, 1, 2):
            assert emu(q, t, 1, mode, 1, 2, 1) == (O.gotoh_rolling(q, t), 0), (q[:8], t[:8], mode)


def test_many_rounds_ring_wraparound(emu):
    # 14 bands on a ring of 3 warps: each warp runs several bands, the last warp feeds the first
    a, b = planted(300, 64 * 14 - 5)
    assert emu(a, b, 1, 0, 1, 3, 1) == (O.gotoh_rolling(a, b), 0)
    assert emu(a, b, 1, 2, 0, 3, 2) == (O.gotoh_rolling(a, b), 0)


@pytest.mark.slow
def test_ring_laps_and_backpressure(emu):
    # T longer than the link ring: entries are overwritten lap after lap, producer must respect progress
    a = rng.random_acgt(400, 0, 150)
    t = rng.random_acgt(400, 1, 9000)
    t[3000:3140] = a[:140]
    assert emu(a, t, 1, 0, 1, 3, 1, link_len=2048) == (O.gotoh_rolling(a, t), 0)


def test_s16_overflow_is_flagged(emu):
    # identical sequences longer than the s16 range cannot be scored in packed 16-bit lanes: the
    # engine must say so (status bit 1) instead of returning a wrapped score
    a = np.frombuffer(b"ACGT" * 82, dtype=np.uint8)
    score, status = emu(a, a, 1, 0, 1, 1, 1, p=(100, -1, 1, 1))
    assert status & 1
    assert emu(a, a, 1, 2, 1, 1, 1, p=(100, -1, 1, 1)) == (100 * 328, 0)


@pytest.mark.parametrize("mode,slack", [(0, 1), (0, 0), (1, 1), (1, 0)])
def test_bottom_boundary_row_of_the_last_band(emu, mode, slack):
    """Stronger than the score: the whole bottom boundary row (H and, affine mode, F at every T position) after
    4 bands must equal the last DP row of the oracle.  Scoring with positive drift (cheap gaps) makes every cell
    matter; this is the check that exposed a missing hand-off of T position 0 with the slack step."""
    p = (3, -2, 2, 2) if mode == 1 else (3, -2, 3, 1)
    for seed in (2010, 2011):
        q = rng.random_acgt(seed, 0, 256)          # 4 bands of 64 rows (R = 1), no padding rows
        t = rng.random_acgt(seed, 1, 300)
        best, H, F = O.gotoh_last_row(t, q, p)     # columns = T positions, last row = last Q row
        score, status, lo, hi = emu(q, t, 1, mode, slack, 3, 1, p, final_row=True)
        assert (score, status) == (best, 0)
        gH = (hi if mode == 1 else lo) + p[2]      # entries carry H - gap_init
        assert gH.tolist() == H[1:].tolist()
        if mode == 0:
            pos = (F[1:] > 0) | (hi > 0)           # non-positive F never matters and conventions differ at the border
            assert hi[pos].tolist() == F[1:][pos].tolist()


@pytest.mark.parametrize("mode", [3, 4])
def test_rebasing_really_triggers(emu, mode):
    """Re-based 16-bit lanes with scores far above the +-8000 trigger (score ~22 000 with match 10): every band re-centres
    several times, publishes its bases in the link rings and translates what it receives; two emulated GPUs in the
    second case.  (The small cases above never leave the first base.)"""
    p = (10, -8, 10, 5) if mode == 3 else (10, -8, 7, 7)
    for n, R, W, G in ((2500, 1, 3, 1), (3000, 2, 2, 2)):
        a = rng.random_acgt(777 + n, 0, n)
        b = rng.mutate(a, 777 + n, 1, 0.05, 0.02)
        want = O.gotoh_rolling(a, b, p)
        assert want > 20000
        for slack in (1, 0):
            assert emu(a, b, R, mode, slack, W, G, p) == (want, 0), (n, R, W, G, slack)


@pytest.mark.parametrize("mode,slack", [(0, 1), (1, 1), (3, 1), (4, 0)])
def test_slack_inside_a_thread(emu, mode, slack):
    """Launch config 4 (HS 1): the hi sub-lane runs two T positions behind the lo sub-lane.  Same cases as the plain
    engine, plus a re-basing one; the lane skew grows to 31*(3+slack)+2 and the table / bottom-row copies are one step
    older, nothing else changes."""
    lin = mode in (1, 4)
    cases = [(300, 1, 2, 1, O.DEFAULT), (800, 2, 3, 2, (3, -2, 2, 2) if lin else (2, -3, 5, 1)), (1000, 4, 2, 1, (1, -3, 1, 1) if lin else (1, -1, 4, 2))]
    for k, (n, R, W, G, p) in enumerate(cases):
        a, b = planted(300 + k, n)
        assert emu(a, b, R, mode, slack, W, G, p, hs=True) == (O.gotoh_rolling(a, b, p), 0), (n, R, W, G, p)
    if mode >= 3:
        p = (10, -8, 7, 7) if lin else (10, -8, 10, 5)
        a = rng.random_acgt(3277, 0, 2500)
        b = rng.mutate(a, 3277, 1, 0.05, 0.02)
        assert emu(a, b, 1, mode, slack, 3, 1, p, hs=True) == (O.gotoh_rolling(a, b, p), 0)


@pytest.mark.parametrize("mode", [3, 4])
def test_rebased_lanes_far_above_zero_run_without_the_floor(emu, mode):
    """Score ~47 000 (match 10): once a band's base passes 30 000 its 256-step blocks run the step loop WITHOUT the clamp
    at the zero floor (swb_engine.cuh: nofloor) -- every band still starts with it, at base 0."""
    p = (10, -8, 10, 5) if mode == 3 else (10, -8, 7, 7)
    a = rng.random_acgt(4242, 0, 5200)
    b = rng.mutate(a, 4242, 1, 0.04, 0.02)
    want = O.gotoh_rolling(a, b, p)
    assert want > 40000
    assert emu(a, b, 4, mode, 0, 2, 2, p) == (want, 0)
    assert emu(a, b, 2, mode, 1, 2, 1, p, hs=True) == (want, 0)


def test_recentring_does_not_wrap_the_stand_in_boundary(emu):
    """LT a multiple of the 256-step block, slack step, base above 30 000: lane 0 holds the stand-in for the boundary
    value of T position LT (-30000 - open) when the band re-centres at the start of its last block; a rising base
    used to wrap it around to +32 5xx, and the pad column scored 66 453 instead of 39 443 (on the GPU: 483 137 instead
    of 456 586 for a 4 M x 4 M pair with 8 rows per sub-lane)."""
    p, n = (10, -8, 7, 7), 4352
    a = rng.random_acgt(1, 0, n)
    b = rng.mutate(a, 1, 1, 0.04, 0.02)[:n]
    b = np.concatenate([b, rng.random_acgt(1, 2, n - len(b))])      # LT = 4352 = 17 * 256 exactly
    assert len(b) == n
    want = O.gotoh_rolling(a, b, p)
    assert want == 39443
    assert emu(a, b, 3, 4, 1, 3, 1, p) == (want, 0)
