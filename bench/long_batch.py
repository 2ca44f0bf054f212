#!/usr/bin/env python
"""Batch scoring of pairs whose shorter side is over 1024 with the multi-band kernel (swb200_batch_score_long,
swb200_score_long_batch) against the per-pair loop these pairs took before (api.score, one swb200_score_ex call each).
Workloads: (1) 20 000 seeded 5 kb pairs, half planted, half random, device-resident; (2) 100 000 cfg5 pairs (10 kb)
generated in HBM, scored without a band and checked against the banded score and, on a sample, swb200_score_ex;
(3) a ragged 1.5-20 kb host mix through swb200_score_long_batch and fasta.score_pairs, against the per-pair loop on a
sample; (4) the crossover: 16 .. 4 096 pairs of 2, 5 and 20 kb, multi-band call against the per-pair loop (timed on up to
`--loop-sample` pairs and scaled to the count).  Device times are CUDA events around the kernel (swb200_last_run).
usage: python bench/long_batch.py [--out FILE] [--quick]   -- one JSON line (also to FILE)"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from concurrentproject_b200 import api, fasta  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="")
ap.add_argument("--quick", action="store_true", help="small sizes (a smoke run of the script)")
ap.add_argument("--loop-sample", type=int, default=24)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/long_batch.py needs a CUDA device")
card = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unknown ({e})"
dev = torch.device("cuda", 0)
ACGT = np.frombuffer(b"ACGT", np.uint8)
Q = a.quick


def pairs(seed, n, lens1, lens2, planted_every=2):
    """Seeded pairs: every planted_every-th one is seq1 with 10 % substitutions (a planted homologue), the rest random."""
    r = np.random.default_rng(seed)
    s1, s2 = [], []
    for k in range(n):
        x = ACGT[r.integers(0, 4, int(lens1[k]))]
        if k % planted_every == 0:
            y = x[:int(lens2[k])].copy()
            if len(y) < lens2[k]:
                y = np.concatenate((y, ACGT[r.integers(0, 4, int(lens2[k]) - len(y))]))
            sub = r.random(len(y)) < 0.10
            y[sub] = ACGT[r.integers(0, 4, int(sub.sum()))]
        else:
            y = ACGT[r.integers(0, 4, int(lens2[k]))]
        s1.append(x.tobytes()); s2.append(y.tobytes())
    return s1, s2


def packed(s1, s2):
    f1, o1, l1 = api._flatten(s1); f2, o2, l2 = api._flatten(s2)
    t = [torch.from_numpy(x).to(dev) for x in (f1, o1, l1, f2, o2, l2)]
    short, long_ = np.minimum(l1, l2), np.maximum(l1, l2)
    pb = api.PackedBatch(ctx, *[x.data_ptr() for x in t], len(s1), int(short.max()), int(long_.max()),
                         int((l1.astype(np.int64) * l2).sum()))
    return pb, t, l1, l2


def device_ms(pb, d, reps=3):
    pb.score_long(d.data_ptr())                       # warm-up of this shape
    ms = []
    for _ in range(reps):
        pb.score_long(d.data_ptr())
        ms.append(ctx.last_run()["engine_ms"])
    return min(ms), ms


def loop_s(s1, s2):
    api.score(s1[0], s2[0])                            # warm-up
    t0 = time.perf_counter()
    got = [api.score(x, y) for x, y in zip(s1, s2)]
    return time.perf_counter() - t0, got


ctx = api.Context(0)
out = {"bench": "long_batch", "card": card, "power_limit": power}

# (1) device-resident throughput: 5 kb pairs
n1 = 2000 if Q else 20000
s1, s2 = pairs(1, n1, np.full(n1, 5000), np.full(n1, 5000))
pb, keep, l1, l2 = packed(s1, s2)
d = torch.empty(n1, dtype=torch.int32, device=dev)
best, all_ms = device_ms(pb, d)
info = ctx.last_run()
cells = int((l1.astype(np.int64) * l2).sum())
band = 64 * info["rows"]
padded = int(sum(-(-min(x, y) // band) * band * (max(x, y) + 63) for x, y in zip(l1.tolist(), l2.tolist())))
sc = d.cpu().numpy()
ls, lg = loop_s(s1[:a.loop_sample], s2[:a.loop_sample])
assert sc[:a.loop_sample].tolist() == lg, "multi-band scores differ from swb200_score_ex"
out["device_5kb"] = {"pairs": n1, "ms": round(best, 2), "ms_all": [round(x, 2) for x in all_ms], "gcups": round(cells / best / 1e6, 1),
                     "padded_cell_fraction": round(1 - cells / padded, 4), "rows": info["rows"], "bands": info["bands"],
                     "warps": info["warps"], "loop_s_per_pair": round(ls / len(lg), 5),
                     "speedup_vs_loop": round(ls / len(lg) * n1 / (best / 1e3), 1), "checksum": int(sc.astype(np.int64).sum())}
pb.close(); del keep
print(json.dumps({"device_5kb": out["device_5kb"]}), flush=True)

# (2) unbanded cfg5: 10 kb pairs generated in HBM; every unbanded score >= the banded one; a sample against swb200_score_ex
n2, L = (5000 if Q else 100000), 10000
d1 = torch.empty(n2 * L, dtype=torch.uint8, device=dev); d2 = torch.empty(n2 * L, dtype=torch.uint8, device=dev)
api.gen_long_pairs_device(0, 5, 0, n2, L, d1.data_ptr(), d2.data_ptr())
off = torch.arange(n2, dtype=torch.int64, device=dev) * L
ln = torch.full((n2,), L, dtype=torch.int32, device=dev)
torch.cuda.synchronize()
pb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n2, L, L, n2 * L * L)
d = torch.empty(n2, dtype=torch.int32, device=dev)
best, all_ms = device_ms(pb, d, reps=2)
unb = d.cpu().numpy()
pb.close()
pbb = api.PackedBatch(ctx, d1.data_ptr(), off.data_ptr(), ln.data_ptr(), d2.data_ptr(), off.data_ptr(), ln.data_ptr(), n2, L, L,
                      n2 * L * 64, keep_order=True)
db = torch.empty(n2, dtype=torch.int32, device=dev)
pbb.score_banded(db.data_ptr(), -32, 31)
banded = db.cpu().numpy()
pbb.close()
samp = np.random.default_rng(2).choice(n2, 200, replace=False)
h1, h2 = d1.view(n2, L), d2.view(n2, L)
ok = all(api.score(h1[k].cpu().numpy(), h2[k].cpu().numpy()) == unb[k] for k in samp.tolist())
out["cfg5_unbanded"] = {"pairs": n2, "ms": round(best, 1), "ms_all": [round(x, 1) for x in all_ms],
                        "gcups": round(n2 * L * L / best / 1e6, 1), "unbanded_ge_banded_all": bool((unb >= banded).all()),
                        "pairs_unbanded_gt_banded": int((unb > banded).sum()), "sample_equal_score_ex": ok,
                        "checksum": int(unb.astype(np.int64).sum())}
del d1, d2
print(json.dumps({"cfg5_unbanded": out["cfg5_unbanded"]}), flush=True)

# (3) host end to end: ragged 1.5-20 kb
n3 = 400 if Q else 4000
r = np.random.default_rng(3)
la = r.integers(1500, 20001, n3); lb = np.minimum(20000, np.maximum(1500, la + r.integers(-3000, 3001, n3)))
s1, s2 = pairs(3, n3, la, lb)
api.score_long_batch(s1[:50], s2[:50])                 # warm-up
t0 = time.perf_counter(); host = api.score_long_batch(s1, s2); t_host = time.perf_counter() - t0
hinfo = api.last_run()
fasta.score_pairs(s1[:50], s2[:50])
t0 = time.perf_counter(); fp = fasta.score_pairs(s1, s2); t_fasta = time.perf_counter() - t0
ls, lg = loop_s(s1[:a.loop_sample], s2[:a.loop_sample])
cells = int((la.astype(np.int64) * lb).sum())
scell = int((la[:a.loop_sample].astype(np.int64) * lb[:a.loop_sample]).sum())
loop_est = ls * cells / scell                           # the loop's time scaled by cells
out["host_ragged"] = {"pairs": n3, "cells": cells, "host_call_s": round(t_host, 3), "host_gcups": round(cells / t_host / 1e9, 1),
                      "host_engine_ms": round(hinfo["engine_ms"], 1), "chunks": hinfo["aux_launches"],
                      "fasta_score_pairs_s": round(t_fasta, 3), "loop_sample_pairs": len(lg), "loop_sample_s": round(ls, 3),
                      "loop_est_s": round(loop_est, 2), "speedup_host_call": round(loop_est / t_host, 1),
                      "speedup_fasta": round(loop_est / t_fasta, 1),
                      "equal": bool(host.tolist() == fp.tolist() and host[:len(lg)].tolist() == lg)}
print(json.dumps({"host_ragged": out["host_ragged"]}), flush=True)

# (4) crossover: multi-band host call against the per-pair loop
cross = []
for L in (2000, 5000, 20000):
    s1, s2 = pairs(4 + L, 4096 if not Q else 256, np.full(4096, L), np.full(4096, L))
    ls, lg = loop_s(s1[:min(a.loop_sample, 16)], s2[:min(a.loop_sample, 16)])
    per = ls / len(lg)
    for n in (16, 64, 256, 1024, 4096):
        if n > len(s1):
            continue
        api.score_long_batch(s1[:n], s2[:n])
        t0 = time.perf_counter(); got = api.score_long_batch(s1[:n], s2[:n]); t = time.perf_counter() - t0
        assert got[:len(lg)].tolist() == lg[:n]
        cross.append({"length": L, "pairs": n, "batch_s": round(t, 4), "loop_s_est": round(per * n, 4), "speedup": round(per * n / t, 2)})
        print(json.dumps(cross[-1]), flush=True)
out["crossover"] = cross
ctx.close()
line = json.dumps(out)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
