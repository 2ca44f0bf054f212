#!/usr/bin/env python
"""Batch alignment on one GPU (swb200_batch_align, swb200_align_batch) against score-only batches and the per-pair
api.align loop, on BASELINE config 4 inputs (150 x 1000, half planted) generated in HBM by swb200_gen_read_pairs_device.
usage: python bench/align_batch.py [--pairs N] [--reps R] [--loop L] [--out FILE]   -- one JSON line (also to FILE)"""
import argparse
import hashlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from concurrentproject_b200 import api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=1_000_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--loop", type=int, default=200, help="pairs of the per-pair api.align loop")
ap.add_argument("--stride", type=int, default=api.OPS_STRIDE)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/align_batch.py needs a CUDA device")

n, L1, L2, seed = a.pairs, 150, 1000, 4
card = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unknown ({e})"

dev = torch.device("cuda", 0)
reads = torch.empty(n * L1, dtype=torch.uint8, device=dev)
wins = torch.empty(n * L2, dtype=torch.uint8, device=dev)
api.gen_read_pairs_device(0, seed, 0, n, L1, L2, reads.data_ptr(), wins.data_ptr())
o1 = torch.arange(n, dtype=torch.int64, device=dev) * L1
o2 = torch.arange(n, dtype=torch.int64, device=dev) * L2
l1 = torch.full((n,), L1, dtype=torch.int32, device=dev)
l2 = torch.full((n,), L2, dtype=torch.int32, device=dev)
torch.cuda.synchronize()

ctx = api.Context(0)
pb = api.PackedBatch(ctx, reads.data_ptr(), o1.data_ptr(), l1.data_ptr(), wins.data_ptr(), o2.data_ptr(), l2.data_ptr(), n, L1, L2,
                     n * L1 * L2)
d_ref = torch.empty(n, dtype=torch.int32, device=dev)
d_sc = torch.empty(n, dtype=torch.int32, device=dev)
d_sp = torch.empty((n, 4), dtype=torch.int32, device=dev)
d_ops = torch.empty((n, a.stride), dtype=torch.int32, device=dev)
d_cnt = torch.empty(n, dtype=torch.int32, device=dev)


def timed(fn):
    fn()                                            # warm-up: module load, scratch buffers grown
    t = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return min(t), t


t_score, _ = timed(lambda: pb.score(d_ref.data_ptr()))
t_align, t_align_all = timed(lambda: pb.align(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), a.stride, d_cnt.data_ptr()))
info = api.last_run(ctx)
scores_equal = bool(torch.equal(d_sc, d_ref))
sc, sp, cnt = d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_cnt.cpu().numpy()
checksum = hashlib.sha256(sc.tobytes() + sp.tobytes()).hexdigest()[:16]

# host end to end: bytes in pinned host memory, copy + pack + align + results back
hr = torch.empty(n * L1, dtype=torch.uint8).pin_memory(); hr.copy_(reads)
hw = torch.empty(n * L2, dtype=torch.uint8).pin_memory(); hw.copy_(wins)
hr, hw = hr.numpy(), hw.numpy()
ho1, ho2 = np.arange(n, dtype=np.int64) * L1, np.arange(n, dtype=np.int64) * L2
hl1, hl2 = np.full(n, L1, np.int32), np.full(n, L2, np.int32)
res = {}


def host():
    res["r"] = api.align_batch_ops(hr, ho1, hl1, hw, ho2, hl2, api.DEFAULT_PARAMS, a.stride)


t_host, _ = timed(host)
host_equal = bool(np.array_equal(res["r"][0], sc) and np.array_equal(res["r"][1], sp) and np.array_equal(res["r"][3], cnt))

# the per-pair loop the batch call replaces
idx = np.random.default_rng(0).choice(n, a.loop, replace=False)
api.align(hr[:L1], hw[:L2])
loop_equal = True
t0 = time.perf_counter()
for k in idx.tolist():
    got = api.align(hr[k * L1:(k + 1) * L1], hw[k * L2:(k + 1) * L2])
    loop_equal &= got[:2] == (int(sc[k]), tuple(int(x) for x in sp[k]))
t_loop = time.perf_counter() - t0
pb.close()
ctx.close()

line = {
    "bench": "align_batch", "card": card, "power_limit": power, "pairs": n, "read_len": L1, "window_len": L2,
    "ops_stride": a.stride, "overflowed": int((cnt < 0).sum()),
    "batch_align_ms": round(t_align * 1e3, 2), "batch_align_ms_all": [round(x * 1e3, 2) for x in t_align_all],
    "batch_align_pairs_per_s": round(n / t_align),
    "batch_score_ms": round(t_score * 1e3, 2), "align_over_score": round(t_align / t_score, 2),
    "host_align_batch_ms": round(t_host * 1e3, 2), "host_align_batch_pairs_per_s": round(n / t_host),
    "loop_pairs": a.loop, "loop_ms": round(t_loop * 1e3, 2), "loop_pairs_per_s": round(a.loop / t_loop, 1),
    "speedup_vs_loop": round((n / t_align) / (a.loop / t_loop), 1),
    "speedup_host_vs_loop": round((n / t_host) / (a.loop / t_loop), 1),
    "cells_three_passes": int(info["cells"]), "launches": int(info["engine_launches"]),
    "scores_equal_batch_score": scores_equal, "host_equal_device": host_equal, "loop_equal": bool(loop_equal),
    "checksum_scores_spans": checksum,
}
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(line) + "\n")
