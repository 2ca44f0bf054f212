#!/usr/bin/env python
"""Banded batches of 64, 128, 256 and 512 diagonals on one GPU, on BASELINE config 5 inputs (100 000 pairs of 10 kb,
seed 5, generated in HBM by swb200_gen_long_pairs_device) with the band centred on the main diagonal.  Per width:
device-resident score time (swb200_batch_score_banded) and in-band cells per second, device-resident alignment time
(swb200_batch_align_banded) and operation-count percentiles, how many pairs score higher than at 64 diagonals and how
many still score below the unbanded score (swb200_batch_score_long), and a checksum of scores, spans and operations.
Device times are CUDA events around the call, the best of --reps after one warm-up call.
usage: python bench/wide_band.py [--pairs N] [--reps R] [--out FILE]   -- one JSON line (also to FILE)"""
import argparse
import hashlib
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from concurrentproject_b200 import api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=100_000)
ap.add_argument("--length", type=int, default=10_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--align-reps", type=int, default=2)
ap.add_argument("--widths", default="64,128,256,512")
ap.add_argument("--stride", type=int, default=api.BANDED_OPS_STRIDE)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/wide_band.py needs a CUDA device")

n, L, seed = a.pairs, a.length, 5
widths = [int(x) for x in a.widths.split(",")]
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


def band_cells(nx, ny, lo, W):
    """In-band cells of an nx x ny rectangle, diagonals lo .. lo + W - 1 of x - y."""
    k = lo + np.arange(W)
    return int(np.clip(np.minimum(ny, nx - k) - np.maximum(1, 1 - k) + 1, 0, None).sum())


def timed(fn, reps):
    """Device time from CUDA events around fn, after one warm-up call: (min, all) in seconds."""
    fn()
    t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1) / 1e3)
    return min(t), t


ctx = api.Context(0)
# the unbanded score of every pair: the multi-band batch kernel on a batch packed with keep_order = 0
pl = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n, L, L,
                     n * L * L)
d_full = torch.empty(n, dtype=torch.int32, device=dev)
pl.score_long(d_full.data_ptr())
torch.cuda.synchronize()
pl.close()
full = d_full.cpu().numpy()

pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n, L, L,
                     n * L * 64, keep_order=True)
d_ref = torch.empty(n, dtype=torch.int32, device=dev)
d_sc = torch.empty(n, dtype=torch.int32, device=dev)
d_sp = torch.empty((n, 4), dtype=torch.int32, device=dev)
d_ops = torch.zeros((n, a.stride), dtype=torch.int32, device=dev)
d_cnt = torch.empty(n, dtype=torch.int32, device=dev)
rows, base = [], None
for W in widths:
    lo, hi = -W // 2, W // 2 - 1
    t_score, t_score_all = timed(lambda: pb.score_banded(d_ref.data_ptr(), lo, hi), a.reps)
    sinfo = api.last_run(ctx)
    t_align, t_align_all = timed(lambda: pb.align_banded(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), a.stride,
                                                         d_cnt.data_ptr(), lo, hi), a.align_reps)
    ainfo = api.last_run(ctx)
    ref, sc, sp, cnt = d_ref.cpu().numpy(), d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_cnt.cpu().numpy()
    ops = d_ops.cpu().numpy().view(np.uint32)
    mask = np.arange(a.stride)[None, :] < np.maximum(cnt, 0)[:, None]
    checksum = hashlib.sha256(ref.tobytes() + sc.tobytes() + sp.tobytes() + cnt.tobytes() + ops[mask].tobytes()).hexdigest()[:16]
    if base is None:
        base = ref.copy()
    cells = n * band_cells(L, L, lo, W)
    rows.append({
        "width": W, "band": [lo, hi],
        "score_ms": round(t_score * 1e3, 2), "score_ms_all": [round(x * 1e3, 2) for x in t_score_all],
        "score_cells": cells, "score_gcups": round(cells / t_score / 1e9, 1), "score_config": int(sinfo["config"]),
        "score_bands": int(sinfo["bands"]),
        "align_ms": round(t_align * 1e3, 2), "align_ms_all": [round(x * 1e3, 2) for x in t_align_all],
        "align_config": int(ainfo["config"]), "align_warps": int(ainfo["warps"]), "align_cells_reported": int(ainfo["cells"]),
        "align_launches": int(ainfo["engine_launches"]),
        "ops_count_p50": int(np.percentile(np.abs(cnt), 50)), "ops_count_p99": int(np.percentile(np.abs(cnt), 99)),
        "ops_count_max": int(np.abs(cnt).max()), "ops_stride": a.stride, "overflowed": int((cnt < 0).sum()),
        "align_scores_equal_score": bool(np.array_equal(sc, ref)),
        "higher_than_w64": int((ref > base).sum()), "lower_than_w64": int((ref < base).sum()),
        "below_unbanded": int((ref < full).sum()), "above_unbanded": int((ref > full).sum()),
        "checksum": checksum,
    })
    print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
pb.close()
ctx.close()

line = {"bench": "wide_band", "card": card, "power_limit": power, "pairs": n, "length": L, "seed": seed,
        "unbanded_checksum": hashlib.sha256(full.tobytes()).hexdigest()[:16], "widths": rows}
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(line) + "\n")
