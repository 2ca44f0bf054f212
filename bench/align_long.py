#!/usr/bin/env python
"""swb200_align on pairs whose traceback directions do not fit in device memory: the 1 000 000 x 1 000 000 pair of
`bench.py --workload n1m` (seed 6), aligned by the blocked traceback, with the time of each phase; and the 100 000 x
100 000 cfg2 pair (seed 2) on both paths, one block and about eight forced blocks, with equal CIGARs asserted.
Times are host clocks around calls that return after a device synchronise: api.align, and api.score_span for passes 1 + 2
alone; pass 3 (forward sweep, recomputes, walks) is the difference.
usage: python bench/align_long.py [--out profiles/r05_align_long.json]   -- one JSON line (also to --out)"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from concurrentproject_b200 import api, rng  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=str(ROOT / "profiles" / "r05_align_long.json"))
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench/align_long.py needs a CUDA device")

card = torch.cuda.get_device_name(0)
sms = torch.cuda.get_device_properties(0).multi_processor_count
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unknown ({e})"


def timed_align(x, y):
    t0 = time.perf_counter()
    r = api.align(x, y)
    return r, time.perf_counter() - t0, api.last_run()["engine_launches"]


def timed_span(x, y):
    """Passes 1 + 2 alone (swb200_score_span: end cell, start cell), host clock around a call that ends in a synchronise."""
    t0 = time.perf_counter()
    api.score_span(x, y)
    return time.perf_counter() - t0


def cigar_ops(c):
    return sum(ch in "=XID" for ch in c)


api.align(rng.random_acgt(9, 0, 3000), rng.random_acgt(9, 1, 3000))     # module load, context, first allocations

# ---- n1m: blocks by itself
x, y = rng.random_acgt(6, 0, 1000000), rng.random_acgt(6, 1, 1000000)
free_before = torch.cuda.mem_get_info(0)[0]
(score, span, cigar), t_n1m, launches = timed_align(x, y)
nb = -(-(span[2] - span[0] + 1) // 256)
blocks = (launches - 1) // 2
t_span = timed_span(x, y)
n1m = {"pair": "n1m 1000000 x 1000000, seed 6", "score": score, "span": list(span), "span_rows": span[2] - span[0] + 1,
       "span_cols": span[3] - span[1] + 1, "bands": nb, "blocks": blocks, "bands_per_block_max": -(-nb // blocks),
       "engine_launches": launches, "cigar_ops": cigar_ops(cigar), "cigar_chars": len(cigar),
       "align_s": round(t_n1m, 3), "passes_1_2_s": round(t_span, 3), "pass_3_s": round(t_n1m - t_span, 3), "free_bytes_before": free_before}
assert score == 114366 and blocks > 1, n1m

# ---- cfg2: one block against about eight
x, y = rng.random_acgt(2, 0, 100000), rng.random_acgt(2, 1, 100000)
api.align(x, y)                                  # warm: directions buffer of the one-block path
(want, t_one, l_one) = timed_align(x, y)
rows = want[1][2] - want[1][0] + 1
k = -(-rows // 8 // 256) * 256
api.configure("align_block_rows", k)
try:
    (got, t_blk, l_blk) = timed_align(x, y)
finally:
    api.configure("align_block_rows", 0)
assert got == want and want[0] == 11446
cfg2 = {"pair": "cfg2 100000 x 100000, seed 2", "score": want[0], "span": list(want[1]), "cigar_ops": cigar_ops(want[2]),
        "one_block_s": round(t_one, 4), "one_block_engine_launches": l_one, "block_rows": k, "blocks": (l_blk - 1) // 2,
        "blocked_s": round(t_blk, 4), "blocked_engine_launches": l_blk, "cigar_equal": True}

line = {"bench": "align_long", "card": card, "power_limit": power, "sms": sms, "n1m": n1m, "cfg2": cfg2}
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(line) + "\n")
