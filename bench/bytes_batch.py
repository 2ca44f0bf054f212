#!/usr/bin/env python
"""Byte batches on one GPU (swb200_batch_pack_device_bytes + swb200_batch_score / swb200_batch_align, and the host calls
swb200_score_batch_bytes / swb200_align_batch_bytes) on BASELINE config 4 inputs (150 x 1000, half planted, generated in
HBM by swb200_gen_read_pairs_device) with one N planted in every read at a position drawn on the host from a seed.
Against: the 2-bit batch calls on the same pairs before the N is planted, the per-pair api.score / api.align loop, and
fasta.score_pairs / align_pairs on a mix with 5 % N reads, routed as now and with the N pairs on the per-pair calls.
usage: python bench/bytes_batch.py [--pairs N] [--reps R] [--loop L] [--mix M] [--out FILE]   -- one JSON line (also to FILE)"""
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
from concurrentproject_b200 import api, fasta  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=1_000_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--loop", type=int, default=200, help="pairs of the per-pair api.score / api.align loops")
ap.add_argument("--mix", type=int, default=100_000, help="pairs of the fasta 5 %% N mix")
ap.add_argument("--stride", type=int, default=api.OPS_STRIDE)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/bytes_batch.py needs a CUDA device")

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


def device_run(byte_symbols):
    """Device-resident score and align of the whole batch: (score s, align s, scores, spans, ops_count, info)."""
    pb = api.PackedBatch(ctx, reads.data_ptr(), o1.data_ptr(), l1.data_ptr(), wins.data_ptr(), o2.data_ptr(), l2.data_ptr(), n, L1,
                         L2, n * L1 * L2, byte_symbols=byte_symbols)
    d_ref = torch.empty(n, dtype=torch.int32, device=dev)
    d_sc = torch.empty(n, dtype=torch.int32, device=dev)
    d_sp = torch.empty((n, 4), dtype=torch.int32, device=dev)
    d_ops = torch.empty((n, a.stride), dtype=torch.int32, device=dev)
    d_cnt = torch.empty(n, dtype=torch.int32, device=dev)
    try:
        t_score, all_score = timed(lambda: pb.score(d_ref.data_ptr()))
        score_info = api.last_run(ctx)
        t_align, all_align = timed(lambda: pb.align(d_sc.data_ptr(), d_sp.data_ptr(), d_ops.data_ptr(), a.stride, d_cnt.data_ptr()))
        align_info = api.last_run(ctx)
    finally:
        pb.close()
    assert torch.equal(d_ref, d_sc)
    return (t_score, all_score, t_align, all_align, d_sc.cpu().numpy(), d_sp.cpu().numpy(), d_cnt.cpu().numpy(), score_info,
            align_info)


def host_run(hr, hw, byte_symbols):
    """End to end from pinned host buffers: copy + pack + kernels + results back."""
    ho1, ho2 = np.arange(n, dtype=np.int64) * L1, np.arange(n, dtype=np.int64) * L2
    hl1, hl2 = np.full(n, L1, np.int32), np.full(n, L2, np.int32)
    res = {}
    score = api.score_batch_bytes_flat if byte_symbols else api.score_batch_flat
    align = api.align_batch_bytes_ops if byte_symbols else api.align_batch_ops
    t_s, _ = timed(lambda: res.__setitem__("s", score(hr, ho1, hl1, hw, ho2, hl2)))
    t_a, _ = timed(lambda: res.__setitem__("a", align(hr, ho1, hl1, hw, ho2, hl2, api.DEFAULT_PARAMS, a.stride)))
    return t_s, t_a, res["s"], res["a"]


def pinned(t):
    h = torch.empty(t.numel(), dtype=torch.uint8).pin_memory()
    h.copy_(t)
    return h.numpy()


def digest(*arrays):
    return hashlib.sha256(b"".join(np.ascontiguousarray(x).tobytes() for x in arrays)).hexdigest()[:16]


# ---- 2-bit calls on the pairs before the N is planted ----
two = device_run(False)
hr0, hw = pinned(reads), pinned(wins)
two_host = host_run(hr0, hw, False)
# ---- one N per read, position from a host seed ----
pos = np.random.default_rng(9).integers(0, L1, n)
reads[torch.from_numpy(np.arange(n, dtype=np.int64) * L1 + pos).to(dev)] = ord("N")
torch.cuda.synchronize()
with_n = device_run(True)
hr = pinned(reads)
by_host = host_run(hr, hw, True)
host_equal = bool(np.array_equal(by_host[2], with_n[4]) and np.array_equal(by_host[3][0], with_n[4]) and
                  np.array_equal(by_host[3][1], with_n[5]) and np.array_equal(by_host[3][3], with_n[6]))

# ---- the per-pair loops the byte batch replaces ----
idx = np.random.default_rng(0).choice(n, a.loop, replace=False)
api.score(hr[:L1], hw[:L2]); api.align(hr[:L1], hw[:L2])
loop_equal = True
t0 = time.perf_counter()
for k in idx.tolist():
    loop_equal &= api.score(hr[k * L1:(k + 1) * L1], hw[k * L2:(k + 1) * L2]) == int(with_n[4][k])
t_score_loop = time.perf_counter() - t0
t0 = time.perf_counter()
for k in idx.tolist():
    got = api.align(hr[k * L1:(k + 1) * L1], hw[k * L2:(k + 1) * L2])
    loop_equal &= got[:2] == (int(with_n[4][k]), tuple(int(x) for x in with_n[5][k]))
t_align_loop = time.perf_counter() - t0

# ---- fasta on a 5 % N mix (the other 95 % the reads before the N was planted): now, with the N pairs on a byte batch,
# against the per-pair route those pairs took before byte batches existed ----
m = min(a.mix, n)
keep_n = np.random.default_rng(11).random(m) < 0.05
mix_r = [bytes((hr if keep_n[k] else hr0)[k * L1:(k + 1) * L1]) for k in range(m)]
mix_w = [bytes(hw[k * L2:(k + 1) * L2]) for k in range(m)]
real_plan = fasta.plan_buckets


def per_pair_plan(*args, **kw):
    return [fasta.Bucket("single", 0, b.index) if b.kind == "bytes" else b for b in real_plan(*args, **kw)]


mix = {}
for route in ("bytes", "per_pair"):
    fasta.plan_buckets = real_plan if route == "bytes" else per_pair_plan
    try:
        t_s, _ = timed(lambda: mix.__setitem__("s" + route, fasta.score_pairs(mix_r, mix_w)))
        t_a, _ = timed(lambda: mix.__setitem__("a" + route, fasta.align_pairs(mix_r, mix_w)))
    finally:
        fasta.plan_buckets = real_plan
    mix[route] = (t_s, t_a)
mix_equal = bool(np.array_equal(mix["sbytes"], mix["sper_pair"]) and np.array_equal(mix["abytes"][0], mix["aper_pair"][0]) and
                 np.array_equal(mix["abytes"][1], mix["aper_pair"][1]) and mix["abytes"][2] == mix["aper_pair"][2])
ctx.close()

ms = lambda t: round(t * 1e3, 2)  # noqa: E731
line = {
    "bench": "bytes_batch", "card": card, "power_limit": power, "pairs": n, "read_len": L1, "window_len": L2,
    "ops_stride": a.stride, "n_per_read": 1,
    "bytes_score_ms": ms(with_n[0]), "bytes_score_ms_all": [ms(x) for x in with_n[1]],
    "bytes_align_ms": ms(with_n[2]), "bytes_align_ms_all": [ms(x) for x in with_n[3]],
    "bytes_align_pairs_per_s": round(n / with_n[2]), "bytes_overflowed": int((with_n[6] < 0).sum()),
    "two_bit_score_ms": ms(two[0]), "two_bit_align_ms": ms(two[2]),
    "bytes_over_two_bit_score": round(with_n[0] / two[0], 2), "bytes_over_two_bit_align": round(with_n[2] / two[2], 2),
    "host_bytes_score_ms": ms(by_host[0]), "host_bytes_align_ms": ms(by_host[1]),
    "host_two_bit_score_ms": ms(two_host[0]), "host_two_bit_align_ms": ms(two_host[1]),
    "loop_pairs": a.loop, "loop_score_ms": ms(t_score_loop), "loop_align_ms": ms(t_align_loop),
    "loop_score_ms_per_pair": round(t_score_loop * 1e3 / a.loop, 3), "loop_align_pairs_per_s": round(a.loop / t_align_loop, 1),
    "bytes_score_speedup_vs_loop": round((n / with_n[0]) / (a.loop / t_score_loop), 1),
    "bytes_align_speedup_vs_loop": round((n / with_n[2]) / (a.loop / t_align_loop), 1),
    "mix_pairs": m, "mix_n_pairs": int(keep_n.sum()),
    "mix_score_pairs_ms": ms(mix["bytes"][0]), "mix_score_pairs_per_pair_route_ms": ms(mix["per_pair"][0]),
    "mix_align_pairs_ms": ms(mix["bytes"][1]), "mix_align_pairs_per_pair_route_ms": ms(mix["per_pair"][1]),
    "score_config": int(with_n[7]["config"]), "align_config": int(with_n[8]["config"]),
    "align_cells_three_passes": int(with_n[8]["cells"]),
    "host_equal_device": host_equal, "loop_equal": bool(loop_equal), "mix_routes_equal": mix_equal,
    "checksum_two_bit": digest(two[4], two[5]), "checksum_bytes": digest(with_n[4], with_n[5]),
}
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(line) + "\n")
