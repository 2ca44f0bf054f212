"""ctypes doorway to tests/banded_span_oracle.c, the CPU checker of banded batch alignment (score and span of the best
local alignment inside a band).  Test infrastructure only: the C file is compiled on first use into a temporary
directory that is removed when the process exits, so nothing is written into the source tree."""
from __future__ import annotations

import atexit
import ctypes as C
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

SRC = Path(__file__).resolve().parent / "banded_span_oracle.c"
DEFAULT = (1, -1, 1, 1)
_lib = None


class _Params(C.Structure):
    _fields_ = [("match", C.c_int), ("mismatch", C.c_int), ("gap_init", C.c_int), ("gap_ext", C.c_int)]


def _load():
    global _lib
    if _lib is None:
        work = Path(tempfile.mkdtemp(prefix="swb200_banded_oracle_"))
        atexit.register(shutil.rmtree, work, True)
        so = work / "libbanded_oracle.so"
        cc = "/usr/bin/gcc" if Path("/usr/bin/gcc").exists() else "gcc"
        subprocess.run([cc, "-O2", "-shared", "-fPIC", "-o", str(so), str(SRC)], check=True)
        lib = C.CDLL(str(so))
        U8 = C.POINTER(C.c_ubyte)
        lib.oracle_gotoh_banded_span.argtypes = [U8, U8, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_Params)] + [C.POINTER(C.c_int)] * 4
        lib.oracle_gotoh_banded_span.restype = C.c_int
        _lib = lib
    return _lib


def _u8(a):
    if isinstance(a, str):
        a = a.encode("latin1")
    if isinstance(a, (bytes, bytearray)):
        a = np.frombuffer(bytes(a), dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def gotoh_banded_span(s1, s2, band_lo, band_hi, p=DEFAULT):
    """(score, i_start, j_start, i_end, j_end), 1-based inclusive (i in seq2, j in seq1), of the best local alignment
    inside band_lo <= j - i <= band_hi; all zero for score 0."""
    a, b = _u8(s1), _u8(s2)
    a1, b1 = (a if len(a) else np.zeros(1, np.uint8)), (b if len(b) else np.zeros(1, np.uint8))
    pp = _Params(*[int(x) for x in p])
    v = [C.c_int(0) for _ in range(4)]
    s = _load().oracle_gotoh_banded_span(a1.ctypes.data_as(C.POINTER(C.c_ubyte)), b1.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                         len(a), len(b), int(band_lo), int(band_hi), C.byref(pp), *[C.byref(x) for x in v])
    return (s,) + tuple(x.value for x in v)
