"""Real-data input path (SURVEY.md 8(f) row 3): FASTA reader and length-bucketed batching.

The reference only ever scores hard-coded or rand() strings (TestFileWithGPU.cpp:25-36); its timing.sh:3-8
shows the intended use, a sweep of many database sequences against queries.  This module feeds such data
to the GPU kernels:

* ``read_fasta``      -- one pass over the file with numpy (no per-record Python loop over bases);
* ``plan_buckets``    -- groups pairs by the kernel geometry their SHORTER sequence needs (rows per lane x
                         lanes per pair, swb_batch.cuh) and orders each bucket by the longer length, so the
                         pairs a warp scores side by side stream about the same number of columns;
* ``score_pairs``     -- scores pair k = (seqs1[k], seqs2[k]) for ragged inputs: ACGT pairs whose shorter side
                         is <= 1024 go bucket by bucket through the batch kernel (swb200_score_batch), pairs with
                         other bytes (N, IUPAC codes, amino acids) and the same limits through the byte batch
                         (swb200_batch_pack_device_bytes), which compares bytes exactly like main.cpp:60, longer ACGT
                         pairs, when the batch beats one call per pair (long_batch_pays), through the multi-band
                         batch kernel (swb200_batch_score_long), everything else (a few long pairs, long pairs with
                         other bytes) through the single-pair engine (swb200_score_ex);
* ``search``          -- one query against every record of a database;
* ``align_pairs``     -- score, span and CIGAR of (seqs1[k], seqs2[k]), each as api.align returns it: pairs whose
                         shorter side is <= 1024 through the batch alignment (swb200_batch_align; pairs with other
                         bytes than A,C,G,T on a byte batch), longer ACGT pairs,
                         when the batch beats one call per pair (align_long_batch_pays), through the long-pair batch
                         alignment (swb200_batch_align_long), everything else pair by pair (swb200_align_device).

The residues are uploaded to HBM once per call (torch is the plumbing for device memory); a bucket only ships its
offsets and lengths and is packed and scored where the bytes already are.  There is no CPU scoring path here."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence, Tuple

import numpy as np

from . import api

# capacities of the batch kernel: rows-per-sub-lane choices {2,4,6,8,10,12,16} x 16 / 32 / 64 sub-lanes per pair
BUCKET_EDGES = (32, 64, 96, 128, 160, 192, 256, 320, 384, 512, 640, 768, 1024)
BATCH_MAX_SHORT = 1024
# Cost model of the two routes for pairs whose shorter side is over BATCH_MAX_SHORT, fitted to the crossover of
# bench/long_batch.py (profiles/r06_long_batch.json; one NVIDIA B200, power limit 1000 W).  One single-pair call costs
# LOOP_CALL_S + LOOP_CELL_S per cell (2, 5, 20 kb: 0.13, 0.21, 0.68 ms).  The multi-band call costs LONG_CALL_S plus
# the longer of its tallest pair on one warp (padded cells at LONG_WARP_CUPS) and all padded cells at LONG_GPU_CUPS.
# So a few long pairs stay on the single-pair engine (20 kb: 64 pairs take 0.04 s there, 0.07 s in the batch).
LOOP_CALL_S, LOOP_CELL_S = 1.8e-4, 1.25e-12
LONG_CALL_S, LONG_WARP_CUPS, LONG_GPU_CUPS = 3e-4, 5.9e9, 8.3e12
# The same form for alignment (align_long_batch_pays), fitted to the crossover of bench/align_long_batch.py
# (profiles/r07_align_long_batch.json; one NVIDIA B200, power limit 1000 W).  One single-pair alignment costs
# ALIGN_LOOP_CALL_S + ALIGN_LOOP_CELL_S per cell (12, 38 ms for a 5, 20 kb pair; measured on 16 pairs: 12.8, 8.7 and
# 36.8 ms for 2, 5 and 20 kb, and the per-pair loop varies between runs, so these are fitted to the decisions, not to
# the times).  The long-pair alignment call costs ALIGN_LONG_CALL_S plus the longer of its tallest pair on one warp and
# all padded cells (256-row bands, three passes) on the whole GPU.
ALIGN_LOOP_CALL_S, ALIGN_LOOP_CELL_S = 1.03e-2, 6.9e-11
ALIGN_LONG_CALL_S, ALIGN_LONG_WARP_CUPS, ALIGN_LONG_GPU_CUPS = 2e-3, 4.6e8, 1.0e11
_IS_ACGT = np.zeros(256, dtype=bool)
_IS_ACGT[[ord(c) for c in "ACGT"]] = True


@dataclass
class FastaRecords:
    names: List[str]
    flat: np.ndarray      # uint8, all residues back to back, upper-cased
    offsets: np.ndarray   # int64, start of record k in flat
    lengths: np.ndarray   # int32

    def __len__(self) -> int:
        return len(self.names)

    def seq(self, k: int) -> np.ndarray:
        o = int(self.offsets[k])
        return self.flat[o:o + int(self.lengths[k])]


def parse_fasta(data: bytes) -> FastaRecords:
    """FASTA text -> records.  Header lines start with '>', sequence lines are concatenated, white space and
    '*' terminators are dropped, letters are upper-cased.  Text before the first header is rejected."""
    buf = np.frombuffer(data, dtype=np.uint8)
    if buf.size == 0:
        return FastaRecords([], np.zeros(0, np.uint8), np.zeros(0, np.int64), np.zeros(0, np.int32))
    nl = np.flatnonzero(buf == 10)
    starts = np.concatenate(([0], nl + 1))
    ends = np.concatenate((nl, [buf.size]))
    keep = starts < buf.size
    starts, ends = starts[keep], ends[keep]
    is_hdr = buf[starts] == ord(">")
    if not is_hdr.any():
        raise ValueError("no FASTA header ('>') found")
    first_hdr = int(np.flatnonzero(is_hdr)[0])
    if any(buf[s:e].tobytes().strip() for s, e in zip(starts[:first_hdr], ends[:first_hdr])):
        raise ValueError("sequence data before the first FASTA header")
    names = [buf[s + 1:e].tobytes().decode("latin1").strip() for s, e in zip(starts[is_hdr], ends[is_hdr])]
    # residue mask: everything on non-header lines except white space and '*'
    line_id = np.zeros(buf.size + 1, dtype=np.int32)
    line_id[starts[is_hdr]] += 1
    line_id[np.minimum(ends[is_hdr], buf.size)] -= 1
    in_hdr = np.cumsum(line_id[:-1]) > 0
    residue = ~in_hdr & (buf > 32) & (buf != ord("*"))
    rec_of_byte = np.cumsum(np.bincount(starts[is_hdr], minlength=buf.size)[:buf.size]) - 1
    flat = buf[residue].copy()
    lower = (flat >= ord("a")) & (flat <= ord("z"))
    flat[lower] -= 32
    lengths = np.bincount(rec_of_byte[residue], minlength=len(names)).astype(np.int32)
    offsets = np.zeros(len(names), dtype=np.int64)
    if len(names) > 1:
        offsets[1:] = np.cumsum(lengths[:-1], dtype=np.int64)
    return FastaRecords(names, flat, offsets, lengths)


def read_fasta(path: str) -> FastaRecords:
    with open(path, "rb") as f:
        return parse_fasta(f.read())


def write_fasta(path: str, names: Sequence[str], seqs: Sequence[bytes], width: int = 60) -> None:
    with open(path, "wb") as f:
        for name, s in zip(names, seqs):
            s = bytes(s)
            f.write(b">" + name.encode("latin1") + b"\n")
            for i in range(0, len(s), width):
                f.write(s[i:i + width] + b"\n")


@dataclass
class Bucket:
    kind: str            # "batch": one swb200_score_batch call; "long": one swb200_batch_score_long call;
                         # "bytes": one call on a byte batch (swb200_batch_pack_device_bytes);
                         # "single": one swb200_score_ex call per pair
    cap: int             # capacity class of the shorter side (0 for "long", "bytes" and "single")
    index: np.ndarray    # pair ids, in the order they are handed to the kernel


def long_batch_pays(short: np.ndarray, long_: np.ndarray) -> bool:
    """True when one multi-band batch call over these pairs is expected to beat one single-pair call each."""
    short = np.asarray(short, dtype=np.int64)
    long_ = np.asarray(long_, dtype=np.int64)
    if short.size == 0:
        return False
    band = 64 * 16                                                  # the band height the tallest pairs get
    padded = (-(-short // band) * band * (long_ + 63)).astype(np.float64)
    loop = short.size * LOOP_CALL_S + float((short * long_).sum()) * LOOP_CELL_S
    batch = LONG_CALL_S + max(float(padded.max()) / LONG_WARP_CUPS, float(padded.sum()) / LONG_GPU_CUPS)
    return batch < loop


def align_long_batch_pays(short: np.ndarray, long_: np.ndarray) -> bool:
    """True when one long-pair alignment call (swb200_batch_align_long) over these pairs is expected to beat one
    swb200_align_device call each."""
    short = np.asarray(short, dtype=np.int64)
    long_ = np.asarray(long_, dtype=np.int64)
    if short.size == 0:
        return False
    padded = (3 * -(-short // 256) * 256 * (long_ + 31)).astype(np.float64)
    loop = short.size * ALIGN_LOOP_CALL_S + float((short * long_).sum()) * ALIGN_LOOP_CELL_S
    batch = ALIGN_LONG_CALL_S + max(float(padded.max()) / ALIGN_LONG_WARP_CUPS, float(padded.sum()) / ALIGN_LONG_GPU_CUPS)
    return batch < loop


def plan_buckets(len1: np.ndarray, len2: np.ndarray, acgt_only: np.ndarray, min_bucket: int = 512, match: int = 1, *,
                 pays=long_batch_pays) -> List[Bucket]:
    """Partition pair ids.  Batch buckets are keyed by the capacity class of min(len1, len2); a class with fewer
    than ``min_bucket`` pairs is merged into the next larger one (a launch costs more than the padding).  Inside a
    bucket pairs are ordered by max(len1, len2), longest first.  ACGT pairs with a shorter side over BATCH_MAX_SHORT
    form one "long" bucket, ordered by padded cells, largest first (the multi-band kernel's warps take pairs in this
    order, so the longest pairs start first), when that call beats the single-pair engine (long_batch_pays).  Pairs the 16-bit batch
    kernels cannot hold (match * min(len) > 32766 - match, swb200.cu: check_batch_score) go to the single-pair engine,
    which re-runs in re-based or 32-bit lanes by itself.  ``pays`` judges the "long" bucket: long_batch_pays for
    scoring, align_long_batch_pays for alignment.  Pairs that are not ``acgt_only`` but within the batch limits form one
    "bytes" bucket, ordered like a batch bucket (a byte batch has one kernel for every shorter side up to 1024)."""
    len1 = np.asarray(len1, dtype=np.int64)
    len2 = np.asarray(len2, dtype=np.int64)
    short = np.minimum(len1, len2)
    long_ = np.maximum(len1, len2)
    acgt = np.asarray(acgt_only, dtype=bool)
    fits16 = int(match) * short <= 32766 - int(match)
    in_range = acgt & fits16
    batchable = in_range & (short <= BATCH_MAX_SHORT)
    byte_ids = np.flatnonzero(~acgt & fits16 & (short <= BATCH_MAX_SHORT))
    long_ids = np.flatnonzero(in_range & (short > BATCH_MAX_SHORT))
    if not pays(short[long_ids], long_[long_ids]):
        long_ids = long_ids[:0]
    out: List[Bucket] = []
    edges = np.array(BUCKET_EDGES)
    cls = np.searchsorted(edges, short, side="left")          # first edge >= short
    carry = np.zeros(0, dtype=np.int64)
    for k, cap in enumerate(BUCKET_EDGES):
        ids = np.concatenate((carry, np.flatnonzero(batchable & (cls == k))))
        if ids.size == 0:
            continue
        if ids.size < min_bucket and k + 1 < len(BUCKET_EDGES):
            carry = ids
            continue
        carry = np.zeros(0, dtype=np.int64)
        order = np.argsort(-long_[ids], kind="stable")
        out.append(Bucket("batch", cap, ids[order]))
    if carry.size:
        order = np.argsort(-long_[carry], kind="stable")
        out.append(Bucket("batch", BUCKET_EDGES[-1], carry[order]))
    if long_ids.size:
        band = 64 * 16                                             # the default band height of the tallest pairs
        padded = (-(-short[long_ids] // band) * band) * (long_[long_ids] + 63)
        out.append(Bucket("long", 0, long_ids[np.argsort(-padded, kind="stable")]))
    if byte_ids.size:
        out.append(Bucket("bytes", 0, byte_ids[np.argsort(-long_[byte_ids], kind="stable")]))
    routed = batchable.copy()
    routed[long_ids] = True
    routed[byte_ids] = True
    rest = np.flatnonzero(~routed)
    if rest.size:
        out.append(Bucket("single", 0, rest))
    return out


def _gather(flat: np.ndarray, offsets: np.ndarray, lengths: np.ndarray, ids: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Bytes of records ``ids`` back to back (vectorised ragged gather; host utility, not on the scoring path)."""
    lens = lengths[ids].astype(np.int32)
    total = int(lens.sum())
    new_off = np.zeros(len(ids), dtype=np.int64)
    if len(ids) > 1:
        new_off[1:] = np.cumsum(lens[:-1], dtype=np.int64)
    if total == 0:
        return np.zeros(1, dtype=np.uint8), new_off, lens
    src = np.repeat(offsets[ids] - new_off, lens) + np.arange(total, dtype=np.int64)
    return np.ascontiguousarray(flat[src]), new_off, lens


def _record_is_acgt(flat: np.ndarray, offsets: np.ndarray, lengths: np.ndarray) -> np.ndarray:
    """Host version of the per-record alphabet check (tests; small inputs)."""
    bad = np.flatnonzero(~_IS_ACGT[flat])
    ok = np.ones(len(offsets), dtype=bool)
    if bad.size:
        ok[np.searchsorted(offsets + lengths, bad, side="right")] = False
    return ok


def _device_records(rec: FastaRecords, torch, device):
    """Residues of all records in HBM (uploaded once per call) and which records are pure A,C,G,T."""
    flat = torch.from_numpy(rec.flat if rec.flat.size else np.zeros(1, np.uint8)).to(device, non_blocking=False)
    ok = np.ones(len(rec), dtype=bool)
    if rec.flat.size:
        f = flat[:rec.flat.size]
        bad = torch.nonzero(~((f == 65) | (f == 67) | (f == 71) | (f == 84))).flatten().cpu().numpy()
        if bad.size:
            ok[np.searchsorted(rec.offsets + rec.lengths, bad, side="right")] = False
    return flat, ok


def score_records(a: FastaRecords, ia: np.ndarray, b: FastaRecords, ib: np.ndarray,
                  params: Sequence[int] = api.DEFAULT_PARAMS, *, min_bucket: int = 512, device: int = 0) -> np.ndarray:
    """Score pair k = (a[ia[k]], b[ib[k]]) for index arrays ia, ib.  Returns int32 scores in pair order.
    The residues go to HBM once; every bucket then only ships its offsets and lengths and is packed and scored
    in place (swb200_batch_pack_device / swb200_batch_score; the "bytes" bucket on a byte batch)."""
    import torch
    ia = np.asarray(ia, dtype=np.int64)
    ib = np.asarray(ib, dtype=np.int64)
    if ia.shape != ib.shape:
        raise ValueError("index arrays differ in length")
    scores = np.zeros(len(ia), dtype=np.int32)
    if len(ia) == 0:
        return scores
    if not torch.cuda.is_available():
        raise RuntimeError("concurrentproject_b200.fasta needs a CUDA device; there is no CPU scoring path")
    dev = torch.device("cuda", device)
    ctx = api.Context(device)
    try:
        fa, ok_a = _device_records(a, torch, dev)
        fb, ok_b = (fa, ok_a) if b is a else _device_records(b, torch, dev)
        l1, l2 = a.lengths[ia].astype(np.int32), b.lengths[ib].astype(np.int32)
        o1, o2 = a.offsets[ia].astype(np.int64), b.offsets[ib].astype(np.int64)
        buckets = plan_buckets(l1, l2, ok_a[ia] & ok_b[ib], min_bucket, match=int(params[0]))
        stream = torch.cuda.current_stream(dev).cuda_stream
        for bk in buckets:
            ids = bk.index
            if bk.kind in ("batch", "long", "bytes"):
                bl1, bl2 = l1[ids], l2[ids]
                d_o1 = torch.from_numpy(o1[ids]).to(dev); d_o2 = torch.from_numpy(o2[ids]).to(dev)
                d_l1 = torch.from_numpy(bl1).to(dev); d_l2 = torch.from_numpy(bl2).to(dev)
                d_sc = torch.empty(len(ids), dtype=torch.int32, device=dev)
                short, long_ = np.minimum(bl1, bl2), np.maximum(bl1, bl2)
                cells = int((bl1.astype(np.int64) * bl2).sum())
                pb = api.PackedBatch(ctx, fa.data_ptr(), d_o1.data_ptr(), d_l1.data_ptr(), fb.data_ptr(), d_o2.data_ptr(),
                                     d_l2.data_ptr(), len(ids), int(short.max()), int(long_.max()), cells, stream=stream,
                                     byte_symbols=bk.kind == "bytes")
                try:
                    if bk.kind == "long":
                        pb.score_long(d_sc.data_ptr(), params, stream=stream)
                    else:
                        pb.score(d_sc.data_ptr(), params, stream=stream)
                finally:
                    pb.close()
                scores[ids] = d_sc.cpu().numpy()
            else:
                for pid in ids:
                    i1, i2 = int(ia[pid]), int(ib[pid])
                    scores[pid] = ctx.score_device(fa.data_ptr() + int(a.offsets[i1]), int(a.lengths[i1]),
                                                   fb.data_ptr() + int(b.offsets[i2]), int(b.lengths[i2]), params, stream=stream)
    finally:
        ctx.close()
    return scores


def align_records(a: FastaRecords, ia: np.ndarray, b: FastaRecords, ib: np.ndarray,
                  params: Sequence[int] = api.DEFAULT_PARAMS, *, min_bucket: int = 512, device: int = 0,
                  ops_stride: int = api.OPS_STRIDE):
    """Align pair k = (a[ia[k]], b[ib[k]]): (scores int32[n], spans int32[n, 4], cigars list[str]) in pair order, each
    as api.align returns it.  The buckets of score_records, with the long bucket judged by align_long_batch_pays: batch
    buckets are packed in place and aligned by swb200_batch_align, the bytes bucket on a byte batch by the same call, the
    long bucket by swb200_batch_align_long (pairs that need more than ops_stride, or api.LONG_OPS_STRIDE, operations once
    more with room for len1 + len2); the rest (long pairs with bytes other than A,C,G,T, long pairs where the batch does
    not pay, pairs whose span could not get direction storage) pair by pair through swb200_align_device."""
    import torch
    ia = np.asarray(ia, dtype=np.int64)
    ib = np.asarray(ib, dtype=np.int64)
    if ia.shape != ib.shape:
        raise ValueError("index arrays differ in length")
    n = len(ia)
    scores = np.zeros(n, dtype=np.int32)
    spans = np.zeros((n, 4), dtype=np.int32)
    cigars: List[str] = [""] * n
    if n == 0:
        return scores, spans, cigars
    if not torch.cuda.is_available():
        raise RuntimeError("concurrentproject_b200.fasta needs a CUDA device; there is no CPU alignment path")
    dev = torch.device("cuda", device)
    ctx = api.Context(device)
    try:
        fa, ok_a = _device_records(a, torch, dev)
        fb, ok_b = (fa, ok_a) if b is a else _device_records(b, torch, dev)
        l1, l2 = a.lengths[ia].astype(np.int32), b.lengths[ib].astype(np.int32)
        o1, o2 = a.offsets[ia].astype(np.int64), b.offsets[ib].astype(np.int64)
        # a long pair goes to the batch only if direction storage for its largest possible span (4 bits a cell in
        # 256-row bands) takes at most a quarter of the free device memory
        short = np.minimum(l1, l2).astype(np.int64)
        dir_bytes = -(-short // 256) * (np.maximum(l1, l2).astype(np.int64) + 31) * 128
        fits = (short <= BATCH_MAX_SHORT) | (dir_bytes <= torch.cuda.mem_get_info(dev)[0] // 4)
        buckets = plan_buckets(l1, l2, ok_a[ia] & ok_b[ib] & fits, min_bucket, match=int(params[0]), pays=align_long_batch_pays)
        stream = torch.cuda.current_stream(dev).cuda_stream

        def run(ids, stride, long_pairs=False, byte_symbols=False):
            bl1, bl2 = l1[ids], l2[ids]
            d_o1 = torch.from_numpy(o1[ids]).to(dev); d_o2 = torch.from_numpy(o2[ids]).to(dev)
            d_l1 = torch.from_numpy(bl1).to(dev); d_l2 = torch.from_numpy(bl2).to(dev)
            d_sc = torch.empty(len(ids), dtype=torch.int32, device=dev)
            d_sp = torch.empty((len(ids), 4), dtype=torch.int32, device=dev)
            d_ops = torch.empty((len(ids), stride), dtype=torch.int32, device=dev)
            d_cnt = torch.empty(len(ids), dtype=torch.int32, device=dev)
            short, long_ = np.minimum(bl1, bl2), np.maximum(bl1, bl2)
            cells = int((bl1.astype(np.int64) * bl2).sum())
            pb = api.PackedBatch(ctx, fa.data_ptr(), d_o1.data_ptr(), d_l1.data_ptr(), fb.data_ptr(), d_o2.data_ptr(),
                                 d_l2.data_ptr(), len(ids), int(short.max()), int(long_.max()), cells, stream=stream,
                                 byte_symbols=byte_symbols)
            try:
                align = pb.align_long if long_pairs else pb.align
                align(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), stride, d_cnt.data_ptr(), params, stream=stream)
            finally:
                pb.close()
            return d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_ops.cpu().numpy().view(np.uint32), d_cnt.cpu().numpy()

        for bk in buckets:
            ids = bk.index
            if bk.kind in ("batch", "long", "bytes"):
                lp, by = bk.kind == "long", bk.kind == "bytes"
                sc, sp, ops, cnt = run(ids, api.LONG_OPS_STRIDE if lp else ops_stride, lp, by)
                scores[ids] = sc
                spans[ids] = sp
                for r, pid in enumerate(ids.tolist()):
                    if cnt[r] >= 0:
                        cigars[pid] = api.cigar_string(ops[r, :cnt[r]])
                redo = ids[cnt < 0]
                if len(redo):
                    _, _, ops2, cnt2 = run(redo, int((l1[redo].astype(np.int64) + l2[redo]).max()), lp, by)
                    for r, pid in enumerate(redo.tolist()):
                        cigars[pid] = api.cigar_string(ops2[r, :cnt2[r]])
            else:
                for pid in ids.tolist():
                    i1, i2 = int(ia[pid]), int(ib[pid])
                    if a.lengths[i1] == 0 or b.lengths[i2] == 0:
                        continue                                   # an empty sequence scores 0: span (0,0,0,0), no CIGAR
                    s_, span, cig = ctx.align_device(fa.data_ptr() + int(a.offsets[i1]), int(a.lengths[i1]),
                                                     fb.data_ptr() + int(b.offsets[i2]), int(b.lengths[i2]), params, stream=stream)
                    scores[pid], spans[pid], cigars[pid] = s_, span, cig
    finally:
        ctx.close()
    return scores, spans, cigars


def _as_records(seqs) -> FastaRecords:
    if isinstance(seqs, FastaRecords):
        return seqs
    flat, offs, lens = api._flatten(seqs)
    return FastaRecords([str(k) for k in range(len(lens))], flat, offs, lens)


def score_pairs(seqs1, seqs2, params: Sequence[int] = api.DEFAULT_PARAMS, *, min_bucket: int = 512) -> np.ndarray:
    """Scores of (seqs1[k], seqs2[k]) for ragged lists of byte strings (or two FastaRecords of equal size)."""
    a, b = _as_records(seqs1), _as_records(seqs2)
    if len(a) != len(b):
        raise ValueError("seqs1 and seqs2 differ in length")
    ids = np.arange(len(a), dtype=np.int64)
    return score_records(a, ids, b, ids, params, min_bucket=min_bucket)


def search(query, database, params: Sequence[int] = api.DEFAULT_PARAMS, *, min_bucket: int = 512) -> np.ndarray:
    """Score one query against every record of ``database`` (FastaRecords or a list of byte strings)."""
    q = _as_records([query])
    db = _as_records(database)
    return score_records(q, np.zeros(len(db), dtype=np.int64), db, np.arange(len(db), dtype=np.int64), params,
                         min_bucket=min_bucket)


def align_pairs(seqs1, seqs2, params: Sequence[int] = api.DEFAULT_PARAMS, *, min_bucket: int = 512):
    """(scores, spans, cigars) of (seqs1[k], seqs2[k]) for ragged lists of byte strings (or two FastaRecords of equal size),
    each as api.align returns it (align_records)."""
    a, b = _as_records(seqs1), _as_records(seqs2)
    if len(a) != len(b):
        raise ValueError("seqs1 and seqs2 differ in length")
    ids = np.arange(len(a), dtype=np.int64)
    return align_records(a, ids, b, ids, params, min_bucket=min_bucket)
