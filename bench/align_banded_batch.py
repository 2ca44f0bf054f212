#!/usr/bin/env python
"""Banded batch alignment on one GPU (swb200_batch_align_banded, swb200_align_banded_batch) against the banded
score-only batch, on BASELINE config 5 inputs (10 kb pairs, band -32..31) generated in HBM by swb200_gen_long_pairs_device.
usage: python bench/align_banded_batch.py [--pairs N] [--reps R] [--sample S] [--out FILE]   -- one JSON line (also to FILE)"""
import argparse
import hashlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from concurrentproject_b200 import api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=100_000)
ap.add_argument("--length", type=int, default=10_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--sample", type=int, default=200, help="pairs checked against the C checker and a host re-score")
ap.add_argument("--stride", type=int, default=api.BANDED_OPS_STRIDE)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/align_banded_batch.py needs a CUDA device")

n, L, lo, hi, seed = a.pairs, a.length, -32, 31, 5
card = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unknown ({e})"

dev = torch.device("cuda", 0)
d1 = torch.empty(n * L, dtype=torch.uint8, device=dev)
d2 = torch.empty(n * L, dtype=torch.uint8, device=dev)
api.gen_long_pairs_device(0, seed, 0, n, L, d1.data_ptr(), d2.data_ptr())
off = torch.arange(n, dtype=torch.int64, device=dev) * L
ln = torch.full((n,), L, dtype=torch.int32, device=dev)
torch.cuda.synchronize()


def band_cells(nx, ny, blo):
    """In-band cells of nx x ny rectangles (arrays), diagonals blo .. blo + 63 of x - y."""
    k = blo[:, None] + np.arange(64)[None, :]
    first = np.maximum(1, 1 - k)
    last = np.minimum(ny[:, None], nx[:, None] - k)
    return np.clip(last - first + 1, 0, None).sum(axis=1)


ctx = api.Context(0)
pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n, L, L,
                     n * L * 64, keep_order=True)
d_ref = torch.empty(n, dtype=torch.int32, device=dev)
d_sc = torch.empty(n, dtype=torch.int32, device=dev)
d_sp = torch.empty((n, 4), dtype=torch.int32, device=dev)
d_ops = torch.zeros((n, a.stride), dtype=torch.int32, device=dev)
d_cnt = torch.empty(n, dtype=torch.int32, device=dev)


def timed(fn):
    """Device time from CUDA events around fn, after one warm-up call: (min, all) in seconds."""
    fn()
    t = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1) / 1e3)
    return min(t), t


t_score, t_score_all = timed(lambda: pb.score_banded(d_ref.data_ptr(), lo, hi))
t_align, t_align_all = timed(lambda: pb.align_banded(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), a.stride,
                                                     d_cnt.data_ptr(), lo, hi))
info = api.last_run(ctx)
scores_equal = bool(torch.equal(d_sc, d_ref))
sc, sp, cnt = d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_cnt.cpu().numpy()
ops = d_ops.cpu().numpy().view(np.uint32)
mask = np.arange(a.stride)[None, :] < np.abs(cnt)[:, None]
checksum = hashlib.sha256(sc.tobytes() + sp.tobytes() + cnt.tobytes() + ops[mask].tobytes()).hexdigest()[:16]

# in-band cells per pass, from the lengths and spans
nn = np.full(n, L, np.int64)
c1 = band_cells(nn, nn, np.full(n, lo, np.int64))
ie, je, is_, js = sp[:, 2].astype(np.int64), sp[:, 3].astype(np.int64), sp[:, 0].astype(np.int64), sp[:, 1].astype(np.int64)
pos = sc > 0
c2 = np.where(pos, band_cells(je, ie, (je - ie) - hi), 0)
c3 = np.where(pos, band_cells(je - js + 1, ie - is_ + 1, lo - (js - is_)), 0)

# host end to end: bytes in pinned host memory, copy + pack + align + results back
h1 = torch.empty(n * L, dtype=torch.uint8).pin_memory(); h1.copy_(d1)
h2 = torch.empty(n * L, dtype=torch.uint8).pin_memory(); h2.copy_(d2)
h1, h2 = h1.numpy(), h2.numpy()
ho, hl = np.arange(n, dtype=np.int64) * L, np.full(n, L, np.int32)
res = {}


def host():
    res["r"] = api.align_banded_batch_ops(h1, ho, hl, h2, ho, hl, lo, hi, api.DEFAULT_PARAMS, a.stride)


host()
t_host_all = []
for _ in range(a.reps):
    t0 = time.perf_counter()
    host()
    t_host_all.append(time.perf_counter() - t0)
t_host = min(t_host_all)
r = res["r"]
host_equal = bool(np.array_equal(r[0], sc) and np.array_equal(r[1], sp) and np.array_equal(r[3], cnt) and np.array_equal(r[2], ops))

# sampled pairs against the C checker and a host re-score of their CIGARs
import banded_oracle as BO  # noqa: E402
from test_gpu_align_banded import check_cigar  # noqa: E402
sample_ok, checked = True, 0
for k in np.random.default_rng(0).choice(n, min(a.sample, n), replace=False).tolist():
    x, y = h1[k * L:(k + 1) * L], h2[k * L:(k + 1) * L]
    want = BO.gotoh_banded_span(x, y, lo, hi)
    if cnt[k] >= 0:
        cig = api.cigar_string(ops[k, :cnt[k]])
    else:
        cig = api.align_banded_batch([bytes(x)], [bytes(y)], lo, hi, ops_stride=2 * L)[2][0]
    ok = (int(sc[k]),) + tuple(int(v) for v in sp[k]) == want and check_cigar(cig, x, y, sp[k], api.DEFAULT_PARAMS, lo, hi) == (want[0], True, True)
    sample_ok &= ok
    checked += 1
pb.close()
ctx.close()

line = {
    "bench": "align_banded_batch", "card": card, "power_limit": power, "pairs": n, "length": L, "band": [lo, hi],
    "ops_stride": a.stride, "overflowed": int((cnt < 0).sum()), "overflow_share": round(float((cnt < 0).mean()), 5),
    "ops_count_p50": int(np.percentile(np.abs(cnt), 50)), "ops_count_p99": int(np.percentile(np.abs(cnt), 99)),
    "ops_count_max": int(np.abs(cnt).max()),
    "batch_align_banded_ms": round(t_align * 1e3, 2), "batch_align_banded_ms_all": [round(x * 1e3, 2) for x in t_align_all],
    "batch_align_banded_pairs_per_s": round(n / t_align),
    "batch_score_banded_ms": round(t_score * 1e3, 2), "batch_score_banded_ms_all": [round(x * 1e3, 2) for x in t_score_all],
    "align_over_score": round(t_align / t_score, 2),
    "host_align_banded_batch_ms": round(t_host * 1e3, 2), "host_align_banded_batch_pairs_per_s": round(n / t_host),
    "cells_pass1": int(c1.sum()), "cells_pass2": int(c2.sum()), "cells_pass3": int(c3.sum()),
    "cells_reported": int(info["cells"]), "launches": int(info["engine_launches"]), "warps": int(info["warps"]),
    "align_gcups_all_passes": round(float(c1.sum() + c2.sum() + c3.sum()) / t_align / 1e9, 1),
    "score_gcups": round(float(c1.sum()) / t_score / 1e9, 1),
    "scores_equal_batch_score_banded": scores_equal, "host_equal_device": host_equal,
    "sample_checked": checked, "sample_ok": bool(sample_ok), "checksum": checksum,
}
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(line) + "\n")
