"""The multi-band batch kernel body (csrc/swb_batch.cuh, batch_warp with LONG) runs on CPU threads
(tests/emu/long_batch_emu.cu, one pthread per lane, two emulated warps sharing one pair counter) against the oracle:
the same source the sm_100a kernels compile.  R = 2 and 4 give bands of 128 and 256 rows, so pairs of a few hundred
rows cross several band edges.  Needs nvcc (host compile only)."""
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

EMU_DIR = Path(__file__).resolve().parent / "emu"
EMU = EMU_DIR / "long_batch_emu"
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")
PARAMS = ((O.DEFAULT, 1), (O.DEFAULT, 0), ((2, -3, 5, 1), 0), ((3, -2, 2, 2), 1), ((2, -1, 1, 3), 0))


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    src = EMU_DIR / "long_batch_emu.cu"
    hdrs = list((EMU_DIR.parent.parent / "concurrentproject_b200" / "csrc").glob("swb_*.cuh"))
    if not EMU.exists() or EMU.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(EMU), str(src),
                        "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("long_batch_emu")

    def run(s1, s2, R, mode, p=O.DEFAULT):
        f = work / "pairs.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(EMU), str(f), str(R), str(mode), *map(str, p)], capture_output=True, text=True,
                             timeout=900, check=True).stdout
        return [int(x) for x in res.split()[1:]]
    return run


def _shapes(seed, band):
    """Short sides at, just below and just above band edges and up to 7 band edges, long sides from shorter than the
    63-step lane skew to a few hundred beyond the short side, empty sequences, planted and random pairs, both orders;
    more pairs than the two emulated warps."""
    r = np.random.default_rng(seed)
    shorts = [band, band - 1, band + 1, 2 * band, 2 * band + 1, 3 * band - 1, int(3.5 * band), 7 * band + 3, 0, 5, 40, band // 2]
    s1, s2 = [], []
    for k, q in enumerate(shorts):
        t = q + 10 if 0 < q <= 40 else (max(q, int(r.integers(q, q + 300))) if k % 4 else max(q, 30))   # long side < 63
        a = rng.random_acgt(seed, 2 * k, t)
        if k % 2 == 0 and q > 4:
            o = int(r.integers(0, t - q + 1))
            b = rng.mutate(a[o:o + q], seed, 2 * k + 1, 0.08, 0.03)[:q]
        else:
            b = rng.random_acgt(seed, 2 * k + 1, q)
        pair = (bytes(b), bytes(a)) if k % 3 else (bytes(a), bytes(b))          # both orders
        s1.append(pair[0]); s2.append(pair[1])
    s1.append(b""); s2.append(b"")
    return s1, s2


@pytest.mark.parametrize("R", [2, 4])
def test_long_batch_kernel_body(emu, R):
    s1, s2 = _shapes(50 + R, 64 * R)
    for p, mode in PARAMS:
        assert emu(s1, s2, R, mode, p) == O.gotoh_batch(s1, s2, p).tolist(), (R, p, mode)


@pytest.mark.parametrize("mode", [0, 1])
def test_vertical_gap_across_a_band_edge(emu, mode):
    """The best path opens a vertical gap in one band and closes it in the next, so the carried F (affine) or H decides."""
    a = rng.random_acgt(71, 0, 600)
    # rows 0..239 match a[0:240], then 30 inserted rows straddling row 256 (R = 4: the band edge), then a[240:600] again
    ins = rng.random_acgt(71, 1, 30)
    b = np.concatenate((a[:240], ins, a[240:560]))
    s1, s2 = [bytes(b)], [bytes(a)]
    for p in ((2, -3, 5, 1), (3, -2, 2, 2), O.DEFAULT):
        if mode == 1 and p[2] != p[3]:
            continue
        want = O.gotoh_batch(s1, s2, p).tolist()
        assert emu(s1, s2, 4, mode, p) == want, (p, mode)
        assert emu(s1, s2, 2, mode, p) == want, (p, mode)
