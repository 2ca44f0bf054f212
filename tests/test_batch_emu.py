"""The batch kernel body (csrc/swb_batch.cuh) and the banded kernel body (csrc/swb_banded.cuh) run on CPU threads
(tests/emu/batch_emu.cu, one pthread per lane) against the oracle: the same source the sm_100a kernels compile.
Needs nvcc (host compile only)."""
import shutil
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
from concurrentproject_b200 import rng

EMU_DIR = Path(__file__).resolve().parent / "emu"
EMU = EMU_DIR / "batch_emu"
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    src = EMU_DIR / "batch_emu.cu"
    hdrs = list((EMU_DIR.parent.parent / "concurrentproject_b200" / "csrc").glob("swb_*.cuh"))
    if not EMU.exists() or EMU.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(EMU), str(src),
                        "-lpthread"], check=True, cwd=EMU_DIR)
    work = tmp_path_factory.mktemp("batch_emu")       # per run: concurrent runs and other users do not collide

    def run(s1, s2, kind, R, mode, G, p=O.DEFAULT, band_lo=-32, tmp=work):
        f = tmp / "swb_batch_emu.bin"
        with open(f, "wb") as out:
            out.write(struct.pack("<i", len(s1)))
            for a, b in zip(s1, s2):
                out.write(struct.pack("<ii", len(a), len(b))); out.write(bytes(a)); out.write(bytes(b))
        res = subprocess.run([str(EMU), str(f), kind, *map(str, [R, mode, G, *p, band_lo])], capture_output=True, text=True,
                             timeout=900, check=True).stdout
        return [int(x) for x in res.split()[1:]]
    return run


def _pairs(seed, npairs, max_read, max_win):
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
        s1.append(bytes(rd)); s2.append(bytes(w))
    return s1, s2


@pytest.mark.parametrize("R,G,max_read", [(2, 8, 32), (4, 8, 64), (10, 8, 150), (4, 16, 120), (2, 32, 110)])
def test_batch_kernel_body(emu, R, G, max_read):
    s1, s2 = _pairs(40 + R + G, 11, max_read, 260)        # 11 pairs: the last group of a warp is partly empty
    for p, mode in ((O.DEFAULT, 1), (O.DEFAULT, 0), ((2, -3, 5, 1), 0), ((3, -2, 2, 2), 1), ((2, -1, 1, 3), 0)):
        assert emu(s1, s2, "batch", R, mode, G, p) == O.gotoh_batch(s1, s2, p).tolist(), (R, G, p, mode)


@pytest.mark.parametrize("G", [16, 8, 4, 2])
def test_banded_kernel_body(emu, G):
    """The four layouts of the banded kernel: 16 threads per pair with two register sets, 8 with four, 4 with eight, 2 with sixteen."""
    r = np.random.default_rng(9)
    a = [bytes(rng.random_acgt(60, k, int(r.integers(1, 420)))) for k in range({4: 11, 2: 19}.get(G, 7))]
    b = [bytes(rng.mutate(np.frombuffer(x, np.uint8), 60, 100 + k, 0.08, 0.03)) if k % 3 else bytes(rng.random_acgt(61, k, 300))
         for k, x in enumerate(a)]
    for lo in (-32, -5, 0, -60, 17):
        for p, mode in ((O.DEFAULT, 1), (O.DEFAULT, 0), ((2, -3, 5, 1), 0), ((3, -2, 3, 1), 0), ((3, -2, 2, 2), 1)):
            want = O.gotoh_banded_batch(a, b, lo, lo + 63, p).tolist()
            assert emu(a, b, "banded", 0, mode, G, p, band_lo=lo) == want, (lo, p, mode, G)
    if G == 4:      # the default layout refills its rings from rolling 64-bit windows whose bit offset follows band_lo: more offsets
        for lo in (-33, -1, -63, 11):
            for p, mode in ((O.DEFAULT, 1), ((2, -3, 5, 1), 0)):
                want = O.gotoh_banded_batch(a, b, lo, lo + 63, p).tolist()
                assert emu(a, b, "banded", 0, mode, G, p, band_lo=lo) == want, (lo, p, mode, G)
