"""ctypes binding of concurrentproject_b200/lib/libswb200.so (C ABI: include/swb200.h, include/algoGPU.h).

There is deliberately no fallback: if the CUDA library is missing or cannot be loaded, importing the
API fails loudly.  Nothing in this package computes a score on the CPU."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["SWB200_LIB"]) if os.environ.get("SWB200_LIB") else PKG / "lib" / "libswb200.so"   # SWB200_LIB: measurement builds (bench/knock.sh)


class Params(C.Structure):
    """swb200_params: MATCH / MISMATCH / G_INIT / G_EXT of the reference (main.cpp:20-23) as data."""
    _fields_ = [("match", C.c_int), ("mismatch", C.c_int), ("gap_init", C.c_int), ("gap_ext", C.c_int)]


class Options(C.Structure):
    _fields_ = [("lanes", C.c_int), ("rows", C.c_int), ("config", C.c_int), ("ctas", C.c_int),
                ("no_linear", C.c_int), ("orient", C.c_int), ("rebase", C.c_int), ("two_sided", C.c_int)]


class RunInfo(C.Structure):
    _fields_ = [("lanes", C.c_int), ("rebased", C.c_int), ("two_sided", C.c_int), ("linear", C.c_int), ("rows", C.c_int), ("config", C.c_int),
                ("ctas", C.c_int), ("warps", C.c_int), ("bands", C.c_int), ("engine_launches", C.c_int),
                ("aux_launches", C.c_int), ("cells", C.c_longlong), ("engine_ms", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


ERRORS = {-1: "CUDA", -2: "ARG", -3: "ALPHABET", -4: "TIMEOUT", -5: "NOMEM", -6: "RANGE"}

U8P = C.POINTER(C.c_ubyte)

# every symbol include/swb200.h and include/algoGPU.h declare
EXPORTS = {
    "swb200_last_error": ([], C.c_char_p),
    "swb200_device_count": ([], C.c_int),
    "swb200_configure": ([C.c_char_p, C.c_char_p], C.c_int),
    "swb200_plan": ([C.c_longlong, C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                     C.POINTER(C.c_double)], C.c_int),
    "swb200_set_devices": ([C.c_int], C.c_int),
    "swb200_get_devices": ([], C.c_int),
    "swb200_score_banded": ([U8P, C.c_int, U8P, C.c_int, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(C.c_int)], C.c_int),
    "swb200_score": ([U8P, C.c_int, U8P, C.c_int, C.POINTER(Params), C.POINTER(C.c_int)], C.c_int),
    "swb200_score_ex": ([U8P, C.c_longlong, U8P, C.c_longlong, C.POINTER(Params), C.POINTER(Options),
                         C.POINTER(C.c_int)], C.c_int),
    "swb200_ctx_create": ([C.c_int, C.POINTER(C.c_void_p)], C.c_int),
    "swb200_ctx_destroy": ([C.c_void_p], None),
    "swb200_score_device": ([C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.POINTER(Params),
                             C.POINTER(Options), C.c_void_p, C.POINTER(C.c_int)], C.c_int),
    "swb200_score_end": ([U8P, C.c_longlong, U8P, C.c_longlong, C.POINTER(Params), C.POINTER(C.c_int),
                          C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)], C.c_int),
    "swb200_score_end_device": ([C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.POINTER(Params),
                                 C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)], C.c_int),
    "swb200_score_span": ([U8P, C.c_longlong, U8P, C.c_longlong, C.POINTER(Params), C.POINTER(C.c_int),
                           C.POINTER(C.c_longlong)], C.c_int),
    "swb200_score_span_device": ([C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.POINTER(Params),
                                  C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_longlong)], C.c_int),
    "swb200_align": ([U8P, C.c_longlong, U8P, C.c_longlong, C.POINTER(Params), C.POINTER(C.c_int), C.POINTER(C.c_longlong),
                      C.c_char_p, C.c_longlong, C.POINTER(C.c_longlong)], C.c_int),
    "swb200_align_device": ([C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.POINTER(Params), C.c_void_p,
                             C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.c_char_p, C.c_longlong, C.POINTER(C.c_longlong)], C.c_int),
    "swb200_last_run": ([C.c_void_p, C.POINTER(RunInfo)], C.c_int),
    "swb200_score_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int),
                            C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_strides": ([C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)], C.c_int),
    "swb200_pack_batch_host": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int),
                                C.c_longlong, C.c_longlong, C.c_longlong, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong),
                                C.POINTER(C.c_int), C.POINTER(C.c_int)], C.c_int),
    "swb200_score_batch_packed": ([C.POINTER(C.c_ulonglong), C.c_longlong, C.POINTER(C.c_ulonglong), C.c_longlong, C.POINTER(C.c_int),
                                   C.POINTER(C.c_int), C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.POINTER(C.c_int)], C.c_int),
    "swb200_banded_strides": ([C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)], C.c_int),
    "swb200_pack_banded_host": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int),
                                 C.c_longlong, C.c_longlong, C.c_longlong, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)], C.c_int),
    "swb200_score_banded_batch_packed": ([C.POINTER(C.c_ulonglong), C.c_longlong, C.POINTER(C.c_ulonglong), C.c_longlong, C.POINTER(C.c_int),
                                          C.POINTER(C.c_int), C.c_longlong, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(Options),
                                          C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_pack_device": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)], C.c_int),
    "swb200_batch_score": ([C.c_void_p, C.POINTER(Params), C.POINTER(Options), C.c_void_p, C.c_void_p], C.c_int),
    "swb200_score_long_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong),
                                 C.POINTER(C.c_int), C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_score_long": ([C.c_void_p, C.POINTER(Params), C.POINTER(Options), C.c_void_p, C.c_void_p], C.c_int),
    "swb200_batch_free": ([C.c_void_p], None),
    "swb200_align_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int),
                            C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.POINTER(C.c_int), C.POINTER(C.c_int),
                            C.POINTER(C.c_uint), C.c_int, C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_align": ([C.c_void_p, C.POINTER(Params), C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_int, C.c_void_p], C.c_int),
    "swb200_align_banded_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong),
                                   C.POINTER(C.c_int), C.c_longlong, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(Options),
                                   C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint), C.c_int, C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_align_banded": ([C.c_void_p, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(Options), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p], C.c_int),
    "swb200_align_long_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong),
                                 C.POINTER(C.c_int), C.c_longlong, C.POINTER(Params), C.POINTER(Options), C.POINTER(C.c_int),
                                 C.POINTER(C.c_int), C.POINTER(C.c_uint), C.c_int, C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_align_long": ([C.c_void_p, C.POINTER(Params), C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_void_p], C.c_int),
    "swb200_score_banded_batch": ([U8P, C.POINTER(C.c_longlong), C.POINTER(C.c_int), U8P, C.POINTER(C.c_longlong),
                                   C.POINTER(C.c_int), C.c_longlong, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(Options),
                                   C.POINTER(C.c_int)], C.c_int),
    "swb200_batch_score_banded": ([C.c_void_p, C.c_int, C.c_int, C.POINTER(Params), C.POINTER(Options), C.c_void_p,
                                   C.c_void_p], C.c_int),
    "swb200_gen_random_device": ([C.c_int, C.c_ulonglong, C.c_ulonglong, C.c_longlong, C.c_void_p, C.c_void_p], C.c_int),
    "swb200_gen_read_pairs_device": ([C.c_int, C.c_ulonglong, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p], C.c_int),
    "swb200_gen_long_pairs_device": ([C.c_int, C.c_ulonglong, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p], C.c_int),
    "swb200_ring_create": ([C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_void_p), C.c_char * 64], C.c_int),
    "swb200_ring_connect": ([C.c_void_p, C.c_char * 64], C.c_int),
    "swb200_ring_connect_local": ([C.c_void_p, C.c_void_p], C.c_int),
    "swb200_ring_connect_root": ([C.c_void_p, C.c_char * 64], C.c_int),
    "swb200_ring_connect_root_local": ([C.c_void_p, C.c_void_p], C.c_int),
    "swb200_ring_combine_pending": ([C.c_void_p], C.c_int),
    "swb200_ring_combine": ([C.c_void_p, C.c_void_p, C.POINTER(C.c_int)], C.c_int),
    "swb200_ring_score_device": ([C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.POINTER(Params),
                                  C.POINTER(Options), C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)], C.c_int),
    "swb200_ring_destroy": ([C.c_void_p], None),
    "SequentialSmithWatermanScoreGPU": ([U8P, U8P, C.c_int, C.c_int], C.c_int),
    "SmithWatermanLazyGPU": ([U8P, U8P, C.c_int, C.c_int], C.c_int),
    "SmithWatermanScoreCUDA": ([U8P, U8P, C.c_int, C.c_int], C.c_int),
    "SmithDiagonalGPU": ([U8P, U8P, C.c_int, C.c_int], C.c_int),
}

_lib = None


def build(jobs: int = 8) -> None:
    """Compile the CUDA library for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    subprocess.run(["make", "-s", f"-j{jobs}", "-C", str(PKG / "csrc")], check=True)


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C concurrentproject_b200/csrc`). There is no CPU fallback.")
        lib = C.CDLL(str(LIB_PATH))
        for name, (argtypes, restype) in EXPORTS.items():
            fn = getattr(lib, name)      # AttributeError here = ABI drift, fail loudly
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


class SwbError(RuntimeError):
    def __init__(self, code: int, where: str):
        msg = load().swb200_last_error().decode(errors="replace")
        super().__init__(f"{where}: SWB200_ERR_{ERRORS.get(code, code)}: {msg}")
        self.code = code
