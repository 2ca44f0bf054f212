#!/usr/bin/env python
"""Batch alignment of pairs whose shorter side is over 1024 (swb200_batch_align_long, swb200_align_long_batch) against
the per-pair loop these pairs took before (api.align, one swb200_align call each).
Workloads: (1) 20 000 seeded 5 kb pairs (the generator of bench/long_batch.py), device-resident: time, cells per pass,
the ratio to swb200_batch_score_long on the same packed batch, the loop on a sample, 200 sampled pairs against
api.align, a checksum and operation-count percentiles; (2) 20 kb pairs whose spans take the pool in several trace
rounds; (3) a ragged 1.5-20 kb host mix through swb200_align_long_batch and fasta.align_pairs against the loop; (4) the
crossover: 16 .. 4 096 pairs of 2, 5 and 20 kb, host call against the loop (timed on up to --loop-sample pairs and
scaled), which fasta.align_long_batch_pays is fitted to.  Device times are CUDA events (swb200_last_run).
usage: python bench/align_long_batch.py [--out FILE] [--quick]   -- one JSON line (also to FILE)"""
import argparse
import json
import subprocess
import sys
import time
import zlib
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
    sys.exit("bench/align_long_batch.py needs a CUDA device")
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
    """bench/long_batch.py's pairs: every planted_every-th one is seq1 with 10 % substitutions, the rest random."""
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


def outputs(n, stride):
    return [torch.zeros(n, dtype=torch.int32, device=dev), torch.zeros((n, 4), dtype=torch.int32, device=dev),
            torch.zeros((n, stride), dtype=torch.int32, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)]


def align_ms(pb, d, stride, reps=3):
    pb.align_long(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), stride, d[3].data_ptr())   # warm-up of this shape
    ms, infos = [], []
    for _ in range(reps):
        pb.align_long(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), stride, d[3].data_ptr())
        infos.append(ctx.last_run())
        ms.append(infos[-1]["engine_ms"])
    return min(ms), ms, infos[-1]


def loop_s(s1, s2):
    api.align(s1[0], s2[0])                            # warm-up
    t0 = time.perf_counter()
    got = [api.align(x, y) for x, y in zip(s1, s2)]
    return time.perf_counter() - t0, got


def as_tuple(sc, sp, ops, cnt, k):
    return (int(sc[k]), tuple(int(x) for x in sp[k]), api.cigar_string(ops[k, :cnt[k]]))


ctx = api.Context(0)
out = {"bench": "align_long_batch", "card": card, "power_limit": power}

# (1) device-resident: 5 kb pairs
n1, stride1 = (2000 if Q else 20000), 8192
s1, s2 = pairs(1, n1, np.full(n1, 5000), np.full(n1, 5000))
pb, keep, l1, l2 = packed(s1, s2)
d = outputs(n1, stride1)
best, all_ms, info = align_ms(pb, d, stride1)
sc, sp, cnt = d[0].cpu().numpy(), d[1].cpu().numpy(), d[3].cpu().numpy()
ops = d[2].cpu().numpy().view(np.uint32)
ds = torch.empty(n1, dtype=torch.int32, device=dev)
pb.score_long(ds.data_ptr())
sms = []
for _ in range(3):
    pb.score_long(ds.data_ptr())
    sms.append(ctx.last_run()["engine_ms"])
assert ds.cpu().numpy().tolist() == sc.tolist(), "scores differ from swb200_batch_score_long"
assert (cnt >= 0).all()
pass1 = int((l1.astype(np.int64) * l2).sum())
pass2 = int((sp[:, 2].astype(np.int64) * sp[:, 3]).sum())
pass3 = int(((sp[:, 2] - sp[:, 0] + 1).astype(np.int64) * (sp[:, 3] - sp[:, 1] + 1) * (sc > 0)).sum())
ls, lg = loop_s(s1[:a.loop_sample], s2[:a.loop_sample])
samp = np.random.default_rng(2).choice(n1, 200, replace=False).tolist()
sample_equal = all(as_tuple(sc, sp, ops, cnt, k) == api.align(s1[k], s2[k]) for k in samp)
crc = 0
for k in range(n1):
    crc = zlib.crc32(ops[k, :cnt[k]].tobytes(), crc)
out["device_5kb"] = {"pairs": n1, "ms": round(best, 2), "ms_all": [round(x, 2) for x in all_ms],
                     "pairs_per_s": round(n1 / (best / 1e3)), "cells_pass1": pass1, "cells_pass2": pass2, "cells_pass3": pass3,
                     "cells_reported": info["cells"], "gcups_all_passes": round((pass1 + pass2 + pass3) / best / 1e6, 1),
                     "bands": info["bands"], "warps_trace": info["warps"], "engine_launches": info["engine_launches"],
                     "score_long_ms": round(min(sms), 2), "ratio_to_score_long": round(best / min(sms), 2),
                     "loop_sample_pairs": len(lg), "loop_s_per_pair": round(ls / len(lg), 5),
                     "loop_est_s": round(ls / len(lg) * n1, 1), "speedup_vs_loop": round(ls / len(lg) * n1 / (best / 1e3), 1),
                     "loop_sample_equal": all(as_tuple(sc, sp, ops, cnt, k) == lg[k] for k in range(len(lg))),
                     "sample200_equal_align": sample_equal,
                     "checksum": {"scores": int(sc.astype(np.int64).sum()), "spans": int(sp.astype(np.int64).sum()), "ops_crc32": crc},
                     "ops_count": {"median": int(np.median(cnt)), "p99": int(np.percentile(cnt, 99)), "max": int(cnt.max()),
                                   "planted_median": int(np.median(cnt[0::2])), "random_median": int(np.median(cnt[1::2]))}}
pb.close(); del keep, d
print(json.dumps({"device_5kb": out["device_5kb"]}), flush=True)

# (2) 20 kb pairs: spans larger than a slot, the pool in rounds
n2, stride2 = (300 if Q else 1000), 16384
s1, s2 = pairs(5, n2, np.full(n2, 20000), np.full(n2, 20000), planted_every=1)
pb, keep, l1, l2 = packed(s1, s2)
d = outputs(n2, stride2)
best, all_ms, info = align_ms(pb, d, stride2, reps=2)
sc, sp, cnt = d[0].cpu().numpy(), d[1].cpu().numpy(), d[3].cpu().numpy()
ops = d[2].cpu().numpy().view(np.uint32)
samp = list(range(0, n2, n2 // 10))
out["device_20kb"] = {"pairs": n2, "ms": round(best, 1), "ms_all": [round(x, 1) for x in all_ms],
                      "pairs_per_s": round(n2 / (best / 1e3), 1), "trace_rounds": info["engine_launches"] - 1,
                      "cells_reported": info["cells"], "sample_equal_align": all(as_tuple(sc, sp, ops, cnt, k) == api.align(s1[k], s2[k]) for k in samp),
                      "ops_count": {"median": int(np.median(cnt)), "p99": int(np.percentile(cnt, 99)), "max": int(cnt.max())},
                      "checksum": int(sc.astype(np.int64).sum())}
pb.close(); del keep, d
print(json.dumps({"device_20kb": out["device_20kb"]}), flush=True)

# (3) host end to end: ragged 1.5-20 kb
n3 = 200 if Q else 2000
r = np.random.default_rng(3)
la = r.integers(1500, 20001, n3); lb = np.minimum(20000, np.maximum(1500, la + r.integers(-3000, 3001, n3)))
s1, s2 = pairs(3, n3, la, lb)
api.align_long_batch(s1[:50], s2[:50])                 # warm-up
t0 = time.perf_counter(); hs, hp, hc = api.align_long_batch(s1, s2); t_host = time.perf_counter() - t0
hinfo = api.last_run()
fasta.align_pairs(s1[:50], s2[:50])
t0 = time.perf_counter(); fs, fp, fc = fasta.align_pairs(s1, s2); t_fasta = time.perf_counter() - t0
ls, lg = loop_s(s1[:a.loop_sample], s2[:a.loop_sample])
cells = int((la.astype(np.int64) * lb).sum())
scell = int((la[:a.loop_sample].astype(np.int64) * lb[:a.loop_sample]).sum())
loop_est = ls * cells / scell                           # the loop's time scaled by cells
host_t = [(int(hs[k]), tuple(int(x) for x in hp[k]), hc[k]) for k in range(n3)]
out["host_ragged"] = {"pairs": n3, "cells": cells, "host_call_s": round(t_host, 3), "host_engine_ms": round(hinfo["engine_ms"], 1),
                      "fasta_align_pairs_s": round(t_fasta, 3), "loop_sample_pairs": len(lg), "loop_sample_s": round(ls, 3),
                      "loop_est_s": round(loop_est, 2), "speedup_host_call": round(loop_est / t_host, 1),
                      "speedup_fasta": round(loop_est / t_fasta, 1),
                      "equal": bool(host_t == [(int(fs[k]), tuple(int(x) for x in fp[k]), fc[k]) for k in range(n3)]
                                    and host_t[:len(lg)] == lg)}
print(json.dumps({"host_ragged": out["host_ragged"]}), flush=True)

# (4) crossover: host call against the per-pair loop
cross = []
for L in (2000, 5000, 20000):
    nmax = 256 if Q else 4096
    s1, s2 = pairs(4 + L, nmax, np.full(nmax, L), np.full(nmax, L))
    ls, lg = loop_s(s1[:min(a.loop_sample, 16)], s2[:min(a.loop_sample, 16)])
    per = ls / len(lg)
    for n in (16, 64, 256, 1024, 4096):
        if n > nmax:
            continue
        api.align_long_batch(s1[:n], s2[:n])
        t0 = time.perf_counter(); got = api.align_long_batch(s1[:n], s2[:n]); t = time.perf_counter() - t0
        assert [(int(got[0][k]), tuple(int(x) for x in got[1][k]), got[2][k]) for k in range(min(n, len(lg)))] == lg[:n]
        cross.append({"length": L, "pairs": n, "batch_s": round(t, 4), "loop_s_est": round(per * n, 4), "speedup": round(per * n / t, 2)})
        print(json.dumps(cross[-1]), flush=True)
out["crossover"] = cross
ctx.close()
line = json.dumps(out)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
