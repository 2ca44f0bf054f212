"""Host-side mirror of the reference's score-function interface, on top of the C ABI.

Same names, argument order and meaning as the reference headers: algoGPU.h:5-9
(``SequentialSmithWatermanScoreGPU``, ``SmithWatermanLazyGPU``, ``SmithWatermanScoreCUDA``: two byte
sequences and their lengths in, the int local-alignment score out) and
SmithDiagonalGPUrefactored.cu:174 (``SmithDiagonalGPU``).  ``score`` adds what the reference keeps
as per-file constants (main.cpp:20-23; README.md:46): MATCH / MISMATCH / GAP_INIT / GAP_EXT.
Everything runs on the GPU through libswb200.so; there is no CPU path here."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from ._lib import Options, Params, RunInfo, SwbError

Bytes = Union[bytes, bytearray, str, np.ndarray]
DEFAULT_PARAMS = (1, -1, 1, 1)  # MATCH, MISMATCH, GAP_INIT, GAP_EXT (main.cpp:20-23)


def _u8(seq: Bytes) -> np.ndarray:
    if isinstance(seq, str):
        seq = seq.encode("latin1")
    if isinstance(seq, (bytes, bytearray)):
        return np.frombuffer(bytes(seq), dtype=np.uint8)
    return np.ascontiguousarray(seq, dtype=np.uint8)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_lib.U8P)


def _params(p) -> Params:
    m, x, gi, ge = p
    return Params(int(m), int(x), int(gi), int(ge))


def _options(lanes=0, rows=0, config=0, ctas=0, no_linear=False, orient=0, rebase=0, two_sided=0) -> Options:
    o = Options()
    o.lanes, o.rows, o.config, o.ctas, o.no_linear, o.orient = lanes, rows, config, ctas, int(bool(no_linear)), orient
    o.rebase, o.two_sided = rebase, two_sided
    return o


def _legacy(name: str, seq1: Bytes, seq2: Bytes, n: Optional[int], m: Optional[int]) -> int:
    a, b = _u8(seq1), _u8(seq2)
    n = len(a) if n is None else n
    m = len(b) if m is None else m
    if n > len(a) or m > len(b):
        raise ValueError("length argument exceeds the buffer")
    return int(getattr(_lib.load(), name)(_ptr(a), _ptr(b), n, m))


def SequentialSmithWatermanScoreGPU(seq1: Bytes, seq2: Bytes, len1: Optional[int] = None, len2: Optional[int] = None) -> int:
    """algoGPU.h:5 / simpleGPU.cu:109."""
    return _legacy("SequentialSmithWatermanScoreGPU", seq1, seq2, len1, len2)


def SmithWatermanLazyGPU(seq1: Bytes, seq2: Bytes, n: Optional[int] = None, m: Optional[int] = None) -> int:
    """algoGPU.h:7 / cudaLazy.cu:58."""
    return _legacy("SmithWatermanLazyGPU", seq1, seq2, n, m)


def SmithWatermanScoreCUDA(seq1: Bytes, seq2: Bytes, n: Optional[int] = None, m: Optional[int] = None) -> int:
    """algoGPU.h:9 / cudaSmithM.cu:128."""
    return _legacy("SmithWatermanScoreCUDA", seq1, seq2, n, m)


def SmithDiagonalGPU(seq1: Bytes, seq2: Bytes, n: Optional[int] = None, m: Optional[int] = None) -> int:
    """SmithDiagonalGPUrefactored.cu:174."""
    return _legacy("SmithDiagonalGPU", seq1, seq2, n, m)


def score(seq1: Bytes, seq2: Bytes, params: Sequence[int] = DEFAULT_PARAMS, *, lanes: int = 0, rows: int = 0,
          config: int = 0, ctas: int = 0, no_linear: bool = False, orient: int = 0, rebase: int = 0, two_sided: int = 0) -> int:
    """Gotoh local-alignment score of two HOST byte sequences with runtime parameters (swb200_score_ex)."""
    a, b = _u8(seq1), _u8(seq2)
    out = C.c_int(0)
    p, o = _params(params), _options(lanes, rows, config, ctas, no_linear, orient, rebase, two_sided)
    rc = _lib.load().swb200_score_ex(_ptr(a), len(a), _ptr(b), len(b), C.byref(p), C.byref(o), C.byref(out))
    if rc != 0:
        raise SwbError(rc, "swb200_score_ex")
    return out.value


def score_end(seq1: Bytes, seq2: Bytes, params: Sequence[int] = DEFAULT_PARAMS) -> Tuple[int, int, int]:
    """(score, i_end, j_end): the score and the 1-based end cell of the best local alignment -- i_end in seq2,
    j_end in seq1; among cells holding the maximum the one with the smallest j_end, then the smallest i_end; (0, 0)
    for score 0 (swb200_score_end).  New relative to the score-only reference (README.md:6)."""
    a, b = _u8(seq1), _u8(seq2)
    out, ie, je = C.c_int(0), C.c_longlong(0), C.c_longlong(0)
    p = _params(params)
    rc = _lib.load().swb200_score_end(_ptr(a), len(a), _ptr(b), len(b), C.byref(p), C.byref(out), C.byref(ie), C.byref(je))
    if rc != 0:
        raise SwbError(rc, "swb200_score_end")
    return out.value, ie.value, je.value


def score_span(seq1: Bytes, seq2: Bytes, params: Sequence[int] = DEFAULT_PARAMS) -> Tuple[int, int, int, int, int]:
    """(score, i_start, j_start, i_end, j_end), 1-based inclusive, i in seq2 and j in seq1: where the best local
    alignment starts and ends (swb200_score_span: end cell by the tracking kernel, start cell by the anchored
    recurrence over the reversed prefixes).  All zero for score 0."""
    a, b = _u8(seq1), _u8(seq2)
    out = C.c_int(0)
    span = (C.c_longlong * 4)()
    p = _params(params)
    rc = _lib.load().swb200_score_span(_ptr(a), len(a), _ptr(b), len(b), C.byref(p), C.byref(out), span)
    if rc != 0:
        raise SwbError(rc, "swb200_score_span")
    return (out.value,) + tuple(int(x) for x in span)


def configure(key: str, value) -> None:
    """Debugging / measurement switches of the library (swb200_configure; include/swb200.h lists the keys)."""
    rc = _lib.load().swb200_configure(key.encode(), str(value).encode())
    if rc != 0:
        raise SwbError(rc, "swb200_configure")


def plan(n: int, m: int, params: Sequence[int] = DEFAULT_PARAMS, lanes: int = 16, sms: int = 148, allow_two_sided: bool = True, **options) -> dict:
    """What the planner would run for an n x m pair on `sms` SMs in all (swb200_plan; needs no GPU): mode, rows per
    sub-lane, launch config (7 = the CTA-chained engine), two-sided sweep, estimated cycles.  lanes: 16 packed 16-bit,
    17 packed 16-bit re-based, 32 = 32-bit lanes."""
    p, o = _params(params), _options(**options)
    out = (C.c_int * 4)()
    est = C.c_double(0.0)
    rc = _lib.load().swb200_plan(n, m, C.byref(p), C.byref(o), lanes, sms, int(allow_two_sided), out, C.byref(est))
    if rc != 0:
        raise SwbError(rc, "swb200_plan")
    return {"mode": out[0], "rows": out[1], "config": out[2], "two_sided": out[3], "est_cycles": est.value}


def last_run(ctx: Optional["Context"] = None) -> dict:
    info = RunInfo()
    rc = _lib.load().swb200_last_run(ctx.handle if ctx else None, C.byref(info))
    if rc != 0:
        raise SwbError(rc, "swb200_last_run")
    return info.as_dict()


class Context:
    """A per-device engine context for sequences that already live in HBM (swb200_ctx_*)."""

    def __init__(self, device: int = 0):
        self.handle = C.c_void_p()
        rc = _lib.load().swb200_ctx_create(device, C.byref(self.handle))
        if rc != 0:
            raise SwbError(rc, "swb200_ctx_create")
        self.device = device

    def close(self):
        if self.handle:
            _lib.load().swb200_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def score_device(self, d_seq1: int, n: int, d_seq2: int, m: int, params: Sequence[int] = DEFAULT_PARAMS, *,
                     stream: int = 0, lanes: int = 0, rows: int = 0, config: int = 0, ctas: int = 0,
                     no_linear: bool = False, orient: int = 0, rebase: int = 0, two_sided: int = 0) -> int:
        """d_seq1/d_seq2: device addresses of raw bytes (e.g. torch_tensor.data_ptr()); stream: cudaStream_t."""
        out = C.c_int(0)
        p, o = _params(params), _options(lanes, rows, config, ctas, no_linear, orient, rebase, two_sided)
        rc = _lib.load().swb200_score_device(self.handle, C.c_void_p(d_seq1), n, C.c_void_p(d_seq2), m, C.byref(p),
                                             C.byref(o), C.c_void_p(stream), C.byref(out))
        if rc != 0:
            raise SwbError(rc, "swb200_score_device")
        return out.value

    def score_end_device(self, d_seq1: int, n: int, d_seq2: int, m: int, params: Sequence[int] = DEFAULT_PARAMS, *,
                         stream: int = 0) -> Tuple[int, int, int]:
        """score_end for sequences resident in HBM (swb200_score_end_device)."""
        out, ie, je = C.c_int(0), C.c_longlong(0), C.c_longlong(0)
        p = _params(params)
        rc = _lib.load().swb200_score_end_device(self.handle, C.c_void_p(d_seq1), n, C.c_void_p(d_seq2), m, C.byref(p),
                                                 C.c_void_p(stream), C.byref(out), C.byref(ie), C.byref(je))
        if rc != 0:
            raise SwbError(rc, "swb200_score_end_device")
        return out.value, ie.value, je.value

    def align_device(self, d_seq1: int, n: int, d_seq2: int, m: int, params: Sequence[int] = DEFAULT_PARAMS, *,
                     stream: int = 0):
        """align for sequences resident in HBM (swb200_align_device): (score, span, cigar) as align returns them."""
        out, need = C.c_int(0), C.c_longlong(0)
        span = (C.c_longlong * 4)()
        p = _params(params)
        cap = 64
        while True:
            buf = C.create_string_buffer(cap)
            rc = _lib.load().swb200_align_device(self.handle, C.c_void_p(d_seq1), n, C.c_void_p(d_seq2), m, C.byref(p),
                                                 C.c_void_p(stream), C.byref(out), span, buf, cap, C.byref(need))
            if rc == -2 and need.value + 1 > cap:            # buffer too small: the call says how much it needs
                cap = need.value + 1
                continue
            if rc != 0:
                raise SwbError(rc, "swb200_align_device")
            return out.value, tuple(int(x) for x in span), buf.value.decode()

    def last_run(self) -> dict:
        return last_run(self)


def _flatten(seqs):
    arrs = [_u8(s) for s in seqs]
    lens = np.array([len(a) for a in arrs], dtype=np.int32)
    offs = np.zeros(len(arrs), dtype=np.int64)
    if len(arrs) > 1:
        offs[1:] = np.cumsum(lens[:-1], dtype=np.int64)
    flat = np.concatenate(arrs) if len(arrs) and int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(flat), offs, lens


def score_batch(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS, *, rows: int = 0, no_linear: bool = False) -> np.ndarray:
    """Scores of many independent HOST pairs in one kernel (swb200_score_batch).  seqs1[k] vs seqs2[k]."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    return score_batch_flat(*_flatten(seqs1), *_flatten(seqs2), params, rows=rows, no_linear=no_linear)


def score_batch_flat(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                     len2: np.ndarray, params: Sequence[int] = DEFAULT_PARAMS, *, rows: int = 0, no_linear: bool = False) -> np.ndarray:
    """swb200_score_batch on already flattened HOST arrays (uint8 bytes, int64 offsets, int32 lengths)."""
    n = len(len1)
    out = np.zeros(n, dtype=np.int32)
    p, o = _params(params), _options(rows=rows, no_linear=no_linear)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_score_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                        off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), C.byref(o),
                                        out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_batch")
    return out


def score_long_batch(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS, *, rows: int = 0, no_linear: bool = False) -> np.ndarray:
    """Scores of many HOST pairs of any size (swb200_score_long_batch): one warp per pair, the shorter side swept in
    bands of 64*rows rows, so pairs whose shorter side is over 1024 stay in one batch kernel."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    return score_long_batch_flat(*_flatten(seqs1), *_flatten(seqs2), params, rows=rows, no_linear=no_linear)


def score_long_batch_flat(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                          len2: np.ndarray, params: Sequence[int] = DEFAULT_PARAMS, *, rows: int = 0,
                          no_linear: bool = False) -> np.ndarray:
    """swb200_score_long_batch on already flattened HOST arrays (uint8 bytes, int64 offsets, int32 lengths)."""
    n = len(len1)
    out = np.zeros(n, dtype=np.int32)
    p, o = _params(params), _options(rows=rows, no_linear=no_linear)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_score_long_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                             off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), C.byref(o),
                                             out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_long_batch")
    return out


def score_banded_batch(seqs1, seqs2, band_lo: int = -32, band_hi: int = 31, params: Sequence[int] = DEFAULT_PARAMS, *,
                       no_linear: bool = False, config: int = 0) -> np.ndarray:
    """Banded scores of many HOST pairs: cell (i, j) counts iff band_lo <= j - i <= band_hi.  The band holds
    band_hi - band_lo + 1 = 64, 128, 256 or 512 diagonals (any other width raises SwbError -2); `config` picks among the
    64-diagonal layouts and is ignored for wider bands."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    return score_banded_batch_flat(*_flatten(seqs1), *_flatten(seqs2), band_lo, band_hi, params, no_linear=no_linear,
                                   config=config)


def score_banded_batch_flat(flat1, off1, len1, flat2, off2, len2, band_lo: int = -32, band_hi: int = 31,
                            params: Sequence[int] = DEFAULT_PARAMS, *, no_linear: bool = False, config: int = 0) -> np.ndarray:
    """swb200_score_banded_batch on already flattened HOST arrays."""
    n = len(len1)
    out = np.zeros(n, dtype=np.int32)
    p, o = _params(params), _options(no_linear=no_linear, config=config)      # config 16: the 16-threads-per-pair layout
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_score_banded_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                               off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, band_lo, band_hi, C.byref(p),
                                               C.byref(o), out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_banded_batch")
    return out


class PackedBatch:
    """A batch packed into the HBM-resident 2-bit format (swb200_batch_*).  All arguments are device addresses.
    byte_symbols=True keeps every byte as it is (swb200_batch_pack_device_bytes: any alphabet, shorter side <= 1024);
    such a batch is scored by score and aligned by align with the byte kernels, and refused by the other calls."""

    def __init__(self, ctx: Context, d_seq1: int, d_off1: int, d_len1: int, d_seq2: int, d_off2: int, d_len2: int, npairs: int,
                 max_short: int, max_long: int, total_cells: int, stream: int = 0, keep_order: bool = False,
                 byte_symbols: bool = False):
        self.ctx, self.npairs = ctx, npairs
        self.handle = C.c_void_p()
        if byte_symbols:
            if keep_order:
                raise ValueError("a byte batch puts the shorter sequence first: keep_order must be False")
            rc = _lib.load().swb200_batch_pack_device_bytes(ctx.handle, C.c_void_p(d_seq1), C.c_void_p(d_off1), C.c_void_p(d_len1),
                                                            C.c_void_p(d_seq2), C.c_void_p(d_off2), C.c_void_p(d_len2), npairs,
                                                            max_short, max_long, total_cells, C.c_void_p(stream),
                                                            C.byref(self.handle))
            if rc != 0:
                raise SwbError(rc, "swb200_batch_pack_device_bytes")
            return
        rc = _lib.load().swb200_batch_pack_device(ctx.handle, C.c_void_p(d_seq1), C.c_void_p(d_off1), C.c_void_p(d_len1),
                                                  C.c_void_p(d_seq2), C.c_void_p(d_off2), C.c_void_p(d_len2), npairs, max_short,
                                                  max_long, total_cells, int(keep_order), C.c_void_p(stream), C.byref(self.handle))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_pack_device")

    def score(self, d_scores: int, params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0, rows: int = 0,
              no_linear: bool = False) -> None:
        p, o = _params(params), _options(rows=rows, no_linear=no_linear)
        rc = _lib.load().swb200_batch_score(self.handle, C.byref(p), C.byref(o), C.c_void_p(stream), C.c_void_p(d_scores))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_score")

    def score_long(self, d_scores: int, params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0, rows: int = 0,
                   no_linear: bool = False) -> None:
        """Scores with the multi-band kernel (swb200_batch_score_long): any shorter side; keep_order=False batches."""
        p, o = _params(params), _options(rows=rows, no_linear=no_linear)
        rc = _lib.load().swb200_batch_score_long(self.handle, C.byref(p), C.byref(o), C.c_void_p(stream), C.c_void_p(d_scores))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_score_long")

    def score_banded(self, d_scores: int, band_lo: int, band_hi: int, params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0,
                     no_linear: bool = False, config: int = 0) -> None:
        p, o = _params(params), _options(no_linear=no_linear, config=config)
        rc = _lib.load().swb200_batch_score_banded(self.handle, band_lo, band_hi, C.byref(p), C.byref(o), C.c_void_p(stream),
                                                   C.c_void_p(d_scores))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_score_banded")

    def align(self, d_scores: int, d_spans: int, d_ops: int, ops_stride: int, d_ops_count: int,
              params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0) -> None:
        """Score, span and alignment operations of every pair (swb200_batch_align; the batch must be packed with
        keep_order=False).  Device outputs: int32 scores[n], int32 spans[n, 4], uint32 ops[n, ops_stride] (count << 4 | op,
        BAM numbering), int32 ops_count[n] (-(count) where ops_stride was too small)."""
        p = _params(params)
        rc = _lib.load().swb200_batch_align(self.handle, C.byref(p), None, C.c_void_p(stream), C.c_void_p(d_scores),
                                            C.c_void_p(d_spans), C.c_void_p(d_ops), ops_stride, C.c_void_p(d_ops_count))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_align")

    def align_banded(self, d_scores: int, d_spans: int, d_ops: int, ops_stride: int, d_ops_count: int, band_lo: int = -32,
                     band_hi: int = 31, params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0) -> None:
        """Score, span and alignment operations of every pair inside the band band_lo <= j - i <= band_hi of 64, 128,
        256 or 512 diagonals (swb200_batch_align_banded; the batch must be packed with keep_order=True).  Device outputs as align writes them."""
        p = _params(params)
        rc = _lib.load().swb200_batch_align_banded(self.handle, band_lo, band_hi, C.byref(p), None, C.c_void_p(stream),
                                                   C.c_void_p(d_scores), C.c_void_p(d_spans), C.c_void_p(d_ops), ops_stride,
                                                   C.c_void_p(d_ops_count))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_align_banded")

    def align_long(self, d_scores: int, d_spans: int, d_ops: int, ops_stride: int, d_ops_count: int,
                   params: Sequence[int] = DEFAULT_PARAMS, *, stream: int = 0) -> None:
        """Score, span and alignment operations of every pair, any shorter side (swb200_batch_align_long; the batch must
        be packed with keep_order=False).  Device outputs as align writes them."""
        p = _params(params)
        rc = _lib.load().swb200_batch_align_long(self.handle, C.byref(p), None, C.c_void_p(stream), C.c_void_p(d_scores),
                                                 C.c_void_p(d_spans), C.c_void_p(d_ops), ops_stride, C.c_void_p(d_ops_count))
        if rc != 0:
            raise SwbError(rc, "swb200_batch_align_long")

    def close(self):
        if self.handle:
            _lib.load().swb200_batch_free(self.handle)
            self.handle = C.c_void_p()


# ---- seeded synthetic inputs generated in HBM (swb200_gen_*_device; host mirror: concurrentproject_b200/rng.py) ----
def gen_random_device(device: int, seed: int, stream_id: int, length: int, d_out: int, stream: int = 0) -> None:
    rc = _lib.load().swb200_gen_random_device(device, seed, stream_id, length, C.c_void_p(d_out), C.c_void_p(stream))
    if rc != 0:
        raise SwbError(rc, "swb200_gen_random_device")


def gen_read_pairs_device(device: int, seed: int, first_pair: int, npairs: int, read_len: int, window_len: int, d_reads: int,
                          d_windows: int, stream: int = 0) -> None:
    """BASELINE config 4 inputs for pairs first_pair .. first_pair+npairs-1 (rng.read_pair per pair)."""
    rc = _lib.load().swb200_gen_read_pairs_device(device, seed, first_pair, npairs, read_len, window_len, C.c_void_p(d_reads),
                                                  C.c_void_p(d_windows), C.c_void_p(stream))
    if rc != 0:
        raise SwbError(rc, "swb200_gen_read_pairs_device")


def gen_long_pairs_device(device: int, seed: int, first_pair: int, npairs: int, length: int, d_seq1: int, d_seq2: int,
                          stream: int = 0) -> None:
    """BASELINE config 5 inputs for pairs first_pair .. first_pair+npairs-1 (rng.long_pair per pair)."""
    rc = _lib.load().swb200_gen_long_pairs_device(device, seed, first_pair, npairs, length, C.c_void_p(d_seq1), C.c_void_p(d_seq2),
                                                  C.c_void_p(stream))
    if rc != 0:
        raise SwbError(rc, "swb200_gen_long_pairs_device")


def set_devices(count: int) -> None:
    """Host-buffer calls (score, score_batch, the four legacy names) use devices 0..count-1 (swb200_set_devices)."""
    rc = _lib.load().swb200_set_devices(count)
    if rc != 0:
        raise SwbError(rc, "swb200_set_devices")


def get_devices() -> int:
    return int(_lib.load().swb200_get_devices())


def align(seq1: Bytes, seq2: Bytes, params: Sequence[int] = DEFAULT_PARAMS):
    """(score, (i_start, j_start, i_end, j_end), cigar): the best local alignment itself (swb200_align).  The extended
    CIGAR reads from the start cell: '=' match, 'X' mismatch, 'I' a base of seq1 against a gap, 'D' a base of seq2 against
    a gap; re-scored with MATCH / MISMATCH / G_INIT + (k-1) G_EXT per gap of length k it gives the score.  A span whose
    traceback directions (half a byte per cell) do not fit in device memory is traced back in blocks of rows, recomputed
    from one stored boundary row per block: same result, about one more sweep over the span.  configure("align_block_rows",
    K) forces blocks of K rows (a multiple of 256)."""
    a, b = _u8(seq1), _u8(seq2)
    out, need = C.c_int(0), C.c_longlong(0)
    span = (C.c_longlong * 4)()
    p = _params(params)
    cap = 64
    while True:
        buf = C.create_string_buffer(cap)
        rc = _lib.load().swb200_align(_ptr(a), len(a), _ptr(b), len(b), C.byref(p), C.byref(out), span, buf, cap, C.byref(need))
        if rc == -2 and need.value + 1 > cap:            # buffer too small: the call says how much it needs
            cap = need.value + 1
            continue
        if rc != 0:
            raise SwbError(rc, "swb200_align")
        return out.value, tuple(int(x) for x in span), buf.value.decode()


def batch_strides(max_short: int, max_long: int) -> Tuple[int, int]:
    qs, ts = C.c_longlong(0), C.c_longlong(0)
    rc = _lib.load().swb200_batch_strides(max_short, max_long, C.byref(qs), C.byref(ts))
    if rc != 0:
        raise SwbError(rc, "swb200_batch_strides")
    return qs.value, ts.value


def pack_batch_host(flat1, off1, len1, flat2, off2, len2):
    """Raw A,C,G,T bytes -> the resident 2-bit layout, on the host (swb200_pack_batch_host): (q_words, q_stride, t_words,
    t_stride, q_len, t_len) as numpy arrays / ints, ready for score_batch_packed."""
    n = len(len1)
    short = np.minimum(len1, len2); long_ = np.maximum(len1, len2)
    qs, ts = batch_strides(int(short.max()) if n else 0, int(long_.max()) if n else 0)
    qw, tw = np.zeros(max(n, 1) * qs, dtype=np.uint64), np.zeros(max(n, 1) * ts, dtype=np.uint64)
    ql, tl = np.zeros(max(n, 1), dtype=np.int32), np.zeros(max(n, 1), dtype=np.int32)
    LL, I, U = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)
    rc = _lib.load().swb200_pack_batch_host(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2), off2.ctypes.data_as(LL),
                                            len2.ctypes.data_as(I), n, qs, ts, qw.ctypes.data_as(U), tw.ctypes.data_as(U),
                                            ql.ctypes.data_as(I), tl.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_pack_batch_host")
    return qw, qs, tw, ts, ql, tl


def score_batch_packed(qw: np.ndarray, q_stride: int, tw: np.ndarray, t_stride: int, ql: np.ndarray, tl: np.ndarray,
                       params: Sequence[int] = DEFAULT_PARAMS, *, rows: int = 0, no_linear: bool = False) -> np.ndarray:
    """swb200_score_batch_packed: HOST batches already in the 2-bit resident format (a quarter of the PCIe bytes)."""
    n = len(ql)
    out = np.zeros(n, dtype=np.int32)
    p, o = _params(params), _options(rows=rows, no_linear=no_linear)
    I, U = C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)
    rc = _lib.load().swb200_score_batch_packed(qw.ctypes.data_as(U), q_stride, tw.ctypes.data_as(U), t_stride, ql.ctypes.data_as(I),
                                               tl.ctypes.data_as(I), n, C.byref(p), C.byref(o), out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_batch_packed")
    return out


def pack_banded_host(flat1, off1, len1, flat2, off2, len2):
    """Raw A,C,G,T bytes -> the resident 2-bit layout for banded scoring (swb200_pack_banded_host; seq1 = columns and
    seq2 = rows keep their roles): (words1, stride1, words2, stride2)."""
    n = len(len1)
    s1, s2 = C.c_longlong(0), C.c_longlong(0)
    rc = _lib.load().swb200_banded_strides(int(len1.max()) if n else 0, int(len2.max()) if n else 0, C.byref(s1), C.byref(s2))
    if rc != 0:
        raise SwbError(rc, "swb200_banded_strides")
    w1, w2 = np.zeros(max(n, 1) * s1.value, dtype=np.uint64), np.zeros(max(n, 1) * s2.value, dtype=np.uint64)
    LL, I, U = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)
    rc = _lib.load().swb200_pack_banded_host(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                             off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, s1.value, s2.value,
                                             w1.ctypes.data_as(U), w2.ctypes.data_as(U))
    if rc != 0:
        raise SwbError(rc, "swb200_pack_banded_host")
    return w1, s1.value, w2, s2.value


def score_banded_batch_packed(w1: np.ndarray, stride1: int, w2: np.ndarray, stride2: int, len1: np.ndarray, len2: np.ndarray,
                              band_lo: int = -32, band_hi: int = 31, params: Sequence[int] = DEFAULT_PARAMS, *,
                              no_linear: bool = False) -> np.ndarray:
    """swb200_score_banded_batch_packed: banded scores of HOST batches already in the 2-bit format (a quarter of the PCIe bytes)."""
    n = len(len1)
    out = np.zeros(n, dtype=np.int32)
    p, o = _params(params), _options(no_linear=no_linear)
    I, U = C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)
    rc = _lib.load().swb200_score_banded_batch_packed(w1.ctypes.data_as(U), stride1, w2.ctypes.data_as(U), stride2,
                                                      len1.ctypes.data_as(I), len2.ctypes.data_as(I), n, band_lo, band_hi,
                                                      C.byref(p), C.byref(o), out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_banded_batch_packed")
    return out


# ---- batch alignment (swb200_align_batch) ----------------------------------------------------------------------------
OPS_STRIDE = 96          # operations per pair in the first attempt: a planted 150-base read needs ~10; on 1 M cfg4 pairs 28 %
                         # (unrelated reads, long gap-rich local alignments) need more and are redone by align_batch
_OP_CHARS = {1: "I", 2: "D", 7: "=", 8: "X"}


def cigar_string(ops) -> str:
    """The extended CIGAR of a row of operations (count << 4 | op, BAM numbering), in align's format."""
    return "".join(f"{int(w) >> 4}{_OP_CHARS[int(w) & 15]}" for w in ops)


def align_batch_ops(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray, len2: np.ndarray,
                    params: Sequence[int] = DEFAULT_PARAMS, ops_stride: int = OPS_STRIDE):
    """swb200_align_batch on flattened HOST arrays: (scores int32[n], spans int32[n, 4], ops uint32[n, ops_stride],
    ops_count int32[n]); ops_count[k] < 0 where pair k needed more than ops_stride operations."""
    n = len(len1)
    scores = np.zeros(n, dtype=np.int32)
    spans = np.zeros((n, 4), dtype=np.int32)
    ops = np.zeros((n, ops_stride), dtype=np.uint32)
    cnt = np.zeros(n, dtype=np.int32)
    p = _params(params)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_align_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                        off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), None,
                                        scores.ctypes.data_as(I), spans.ctypes.data_as(I),
                                        ops.ctypes.data_as(C.POINTER(C.c_uint)), ops_stride, cnt.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_align_batch")
    return scores, spans, ops, cnt


def align_batch(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS, *, ops_stride: int = OPS_STRIDE):
    """(scores int32[n], spans int32[n, 4], cigars list[str]): align(seqs1[k], seqs2[k]) for every pair, in one batch call
    (swb200_align_batch; the limits of score_batch).  Pairs whose alignment needs more than ops_stride operations are
    aligned again in a second batch with room for len1 + len2 operations, which always suffices."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    f1, o1, l1 = _flatten(seqs1)
    f2, o2, l2 = _flatten(seqs2)
    scores, spans, ops, cnt = align_batch_ops(f1, o1, l1, f2, o2, l2, params, ops_stride)
    cigars = [cigar_string(ops[k, :c]) if c >= 0 else None for k, c in enumerate(cnt.tolist())]
    redo = np.flatnonzero(cnt < 0)
    if len(redo):
        stride = int((l1[redo].astype(np.int64) + l2[redo]).max())
        _, _, ops2, cnt2 = align_batch_ops(f1, o1[redo].copy(), l1[redo].copy(), f2, o2[redo].copy(), l2[redo].copy(), params, stride)
        for r, k in enumerate(redo.tolist()):
            cigars[k] = cigar_string(ops2[r, :cnt2[r]])
    return scores, spans, cigars


# ---- byte batches: any bytes, shorter side <= 1024 (swb200_score_batch_bytes, swb200_align_batch_bytes) -------------
def score_batch_bytes(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS) -> np.ndarray:
    """score_batch for pairs in any bytes (N, IUPAC codes, lower case, amino acids): bytes compare as they are, exactly
    as score compares them, in one batch call (swb200_score_batch_bytes; the limits of score_batch without its alphabet)."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    return score_batch_bytes_flat(*_flatten(seqs1), *_flatten(seqs2), params)


def score_batch_bytes_flat(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                           len2: np.ndarray, params: Sequence[int] = DEFAULT_PARAMS) -> np.ndarray:
    """swb200_score_batch_bytes on already flattened HOST arrays (uint8 bytes, int64 offsets, int32 lengths)."""
    n = len(len1)
    out = np.zeros(n, dtype=np.int32)
    p = _params(params)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_score_batch_bytes(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                              off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), None,
                                              out.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_score_batch_bytes")
    return out


def align_batch_bytes_ops(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                          len2: np.ndarray, params: Sequence[int] = DEFAULT_PARAMS, ops_stride: int = OPS_STRIDE):
    """swb200_align_batch_bytes on flattened HOST arrays: (scores, spans, ops, ops_count) as align_batch_ops returns them."""
    n = len(len1)
    scores = np.zeros(n, dtype=np.int32)
    spans = np.zeros((n, 4), dtype=np.int32)
    ops = np.zeros((n, ops_stride), dtype=np.uint32)
    cnt = np.zeros(n, dtype=np.int32)
    p = _params(params)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_align_batch_bytes(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                              off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), None,
                                              scores.ctypes.data_as(I), spans.ctypes.data_as(I),
                                              ops.ctypes.data_as(C.POINTER(C.c_uint)), ops_stride, cnt.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_align_batch_bytes")
    return scores, spans, ops, cnt


def align_batch_bytes(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS, *, ops_stride: int = OPS_STRIDE):
    """(scores int32[n], spans int32[n, 4], cigars list[str]): align(seqs1[k], seqs2[k]) for every pair in any bytes, in
    one batch call (swb200_align_batch_bytes; the limits of align_batch without its alphabet).  Pairs whose alignment
    needs more than ops_stride operations are aligned again with room for len1 + len2 operations."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    f1, o1, l1 = _flatten(seqs1)
    f2, o2, l2 = _flatten(seqs2)
    scores, spans, ops, cnt = align_batch_bytes_ops(f1, o1, l1, f2, o2, l2, params, ops_stride)
    cigars = [cigar_string(ops[k, :c]) if c >= 0 else None for k, c in enumerate(cnt.tolist())]
    redo = np.flatnonzero(cnt < 0)
    if len(redo):
        stride = int((l1[redo].astype(np.int64) + l2[redo]).max())
        _, _, ops2, cnt2 = align_batch_bytes_ops(f1, o1[redo].copy(), l1[redo].copy(), f2, o2[redo].copy(), l2[redo].copy(),
                                                 params, stride)
        for r, k in enumerate(redo.tolist()):
            cigars[k] = cigar_string(ops2[r, :cnt2[r]])
    return scores, spans, cigars


# ---- banded batch alignment (swb200_align_banded_batch) ----------------------------------------------------------------
BANDED_OPS_STRIDE = 3328  # operations per pair in the first attempt.  On 100 000 cfg5 pairs (10 kb, 10 % substitutions,
                          # 2 % indels, band -32..31, default scoring) the alignments need 2 233 operations at the median,
                          # 3 256 at the 99th percentile and 5 910 at most (bench/align_banded_batch.py, NVIDIA B200), so
                          # about 1 % of such pairs are redone.  The ops buffer costs npairs x stride x 4 B: 13 KB per pair,
                          # 1.3 GB for 100 000 pairs.


def align_banded_batch_ops(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                           len2: np.ndarray, band_lo: int = -32, band_hi: int = 31, params: Sequence[int] = DEFAULT_PARAMS,
                           ops_stride: int = BANDED_OPS_STRIDE):
    """swb200_align_banded_batch on flattened HOST arrays: (scores int32[n], spans int32[n, 4], ops uint32[n, ops_stride],
    ops_count int32[n]) as align_batch_ops returns them; ops_count[k] < 0 where pair k needed more than ops_stride."""
    n = len(len1)
    scores = np.zeros(n, dtype=np.int32)
    spans = np.zeros((n, 4), dtype=np.int32)
    ops = np.zeros((n, ops_stride), dtype=np.uint32)
    cnt = np.zeros(n, dtype=np.int32)
    p = _params(params)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_align_banded_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                               off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, band_lo, band_hi, C.byref(p),
                                               None, scores.ctypes.data_as(I), spans.ctypes.data_as(I),
                                               ops.ctypes.data_as(C.POINTER(C.c_uint)), ops_stride, cnt.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_align_banded_batch")
    return scores, spans, ops, cnt


def align_banded_batch(seqs1, seqs2, band_lo: int = -32, band_hi: int = 31, params: Sequence[int] = DEFAULT_PARAMS, *,
                       ops_stride: int = BANDED_OPS_STRIDE):
    """(scores int32[n], spans int32[n, 4], cigars list[str]): the best local alignment of every pair inside the band
    band_lo <= j - i <= band_hi (64, 128, 256 or 512 diagonals), in one batch call (swb200_align_banded_batch; the
    limits of score_banded_batch).  Pairs whose alignment needs more than ops_stride operations are aligned again with room for
    len1 + len2 operations, which always suffices."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    f1, o1, l1 = _flatten(seqs1)
    f2, o2, l2 = _flatten(seqs2)
    scores, spans, ops, cnt = align_banded_batch_ops(f1, o1, l1, f2, o2, l2, band_lo, band_hi, params, ops_stride)
    cigars = [cigar_string(ops[k, :c]) if c >= 0 else None for k, c in enumerate(cnt.tolist())]
    redo = np.flatnonzero(cnt < 0)
    if len(redo):
        stride = int((l1[redo].astype(np.int64) + l2[redo]).max())
        _, _, ops2, cnt2 = align_banded_batch_ops(f1, o1[redo].copy(), l1[redo].copy(), f2, o2[redo].copy(), l2[redo].copy(),
                                                  band_lo, band_hi, params, stride)
        for r, k in enumerate(redo.tolist()):
            cigars[k] = cigar_string(ops2[r, :cnt2[r]])
    return scores, spans, cigars


# ---- long-pair batch alignment (swb200_align_long_batch) --------------------------------------------------------------
LONG_OPS_STRIDE = 4096    # operations per pair in the first attempt.  On 20 000 seeded 5 kb pairs (half planted with 10 %
                          # substitutions, half random; default scoring) the alignments need 1 963 operations at the median,
                          # 3 735 at the 99th percentile and 3 816 at most (bench/align_long_batch.py, NVIDIA B200); 20 kb
                          # planted pairs need 2 875 at the median.  The ops buffer costs 16 KB per pair.


def align_long_batch_ops(flat1: np.ndarray, off1: np.ndarray, len1: np.ndarray, flat2: np.ndarray, off2: np.ndarray,
                         len2: np.ndarray, params: Sequence[int] = DEFAULT_PARAMS, ops_stride: int = LONG_OPS_STRIDE):
    """swb200_align_long_batch on flattened HOST arrays: (scores int32[n], spans int32[n, 4], ops uint32[n, ops_stride],
    ops_count int32[n]) as align_batch_ops returns them; ops_count[k] < 0 where pair k needed more than ops_stride."""
    n = len(len1)
    scores = np.zeros(n, dtype=np.int32)
    spans = np.zeros((n, 4), dtype=np.int32)
    ops = np.zeros((n, ops_stride), dtype=np.uint32)
    cnt = np.zeros(n, dtype=np.int32)
    p = _params(params)
    LL, I = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    rc = _lib.load().swb200_align_long_batch(_ptr(flat1), off1.ctypes.data_as(LL), len1.ctypes.data_as(I), _ptr(flat2),
                                             off2.ctypes.data_as(LL), len2.ctypes.data_as(I), n, C.byref(p), None,
                                             scores.ctypes.data_as(I), spans.ctypes.data_as(I),
                                             ops.ctypes.data_as(C.POINTER(C.c_uint)), ops_stride, cnt.ctypes.data_as(I))
    if rc != 0:
        raise SwbError(rc, "swb200_align_long_batch")
    return scores, spans, ops, cnt


def align_long_batch(seqs1, seqs2, params: Sequence[int] = DEFAULT_PARAMS, *, ops_stride: int = LONG_OPS_STRIDE):
    """(scores int32[n], spans int32[n, 4], cigars list[str]): align(seqs1[k], seqs2[k]) for every pair of any size, in
    one batch call (swb200_align_long_batch; the limits of score_long_batch).  Pairs whose alignment needs more than
    ops_stride operations are aligned again with room for len1 + len2 operations, which always suffices."""
    if len(seqs1) != len(seqs2):
        raise ValueError("seqs1 and seqs2 differ in length")
    f1, o1, l1 = _flatten(seqs1)
    f2, o2, l2 = _flatten(seqs2)
    scores, spans, ops, cnt = align_long_batch_ops(f1, o1, l1, f2, o2, l2, params, ops_stride)
    cigars = [cigar_string(ops[k, :c]) if c >= 0 else None for k, c in enumerate(cnt.tolist())]
    redo = np.flatnonzero(cnt < 0)
    if len(redo):
        stride = int((l1[redo].astype(np.int64) + l2[redo]).max())
        _, _, ops2, cnt2 = align_long_batch_ops(f1, o1[redo].copy(), l1[redo].copy(), f2, o2[redo].copy(), l2[redo].copy(),
                                                params, stride)
        for r, k in enumerate(redo.tolist()):
            cigars[k] = cigar_string(ops2[r, :cnt2[r]])
    return scores, spans, cigars
