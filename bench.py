#!/usr/bin/env python
"""bench.py -- GCUPS of the score-only Smith-Waterman/Gotoh hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|...] [--no-extra]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  The headline workload is BASELINE config 2:
one 100 000 x 100 000 pair of seeded random ACGT (seed 2), parameters 1/-1/1/1, one pair per GPU (weak scaling, no
data-path collective); its score is checked against the committed golden value on every step.  One JSON line goes to
stdout (rank 0):
  value      device-resident GCUPS: inputs already in HBM, CUDA events around each step
             (encode kernels + wavefront kernel + 40-byte result copy), L2 flushed between steps
  e2e        the same metric through the host-buffer C ABI call the reference harness makes
             (algoGPU.h SmithWatermanScoreCUDA): H2D + encode + kernel + D2H, wall clock
  roofline   the wavefront kernel alone against the integer-ALU (DPX) issue-rate roofline of
             SURVEY.md 8d: 148 SMs x f_clk x L x V / 7, L measured by bench/intpeak.cu
  cpu_baseline  the reference's own CPU path (oracle/_ref/libref.so = unmodified
             lazySmith_parallel_threads.cpp) timed on this box's host cores, bounded sample
and, unless --no-extra, two sub-records measured in the same run on the same N GPUs:
  ring       BASELINE config 3: ONE 4 000 000 x 4 000 000 pair over the ring of all N GPUs (strong scaling; the boundary
             stream crosses GPUs inside the kernel, peer stores over NVLink), score checked against the pinned golden
  batch      BASELINE config 4: 10 M read/window pairs generated in HBM by the seeded device generator, sharded
             pair-wise over the N GPUs (strong scaling, no communication), a sample checked against the oracle and a
             64-bit checksum over all scores that is the same for every N
Every timed loop, the sub-records' and the end-to-end host-call figures' included, runs --steps times (after --warmup
untimed steps; at least 3 for pairs and batches, 1 for the ring); the e2e figures are per call.
--workload cfg1|n1m|ring400k|ring1m|cfg3|cfg4|cfg5 makes that workload the line itself.
--impl reference runs only the reference's CPU path, as the reference arm.
--dump-outputs DIR writes, after the timed steps, the scores the timed path returned in its last step: one
DIR/<workload>_scores.npy per record (float64 for single pairs, float32 for batches, exact for every score these
workloads reach), with a .rank<r> suffix when several ranks run.  Inputs are seeded, so two builds of the project
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import sys
import threading
import time
from pathlib import Path

import numpy as np

if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"         # keep NCCL's version banner off stdout: one JSON line is the contract

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from concurrentproject_b200 import rng  # noqa: E402

METRIC = "GCUPS (affine Smith-Waterman score, cells/s/1e9)"
DPX_LANE_INSTR_PER_CLK_PER_SM = 64.0   # L: profiles/r01_intpeak.jsonl (VIMNMX3/VIADDMNMX.S16x2 streams, B200)
INSTR_PER_CELL_VECTOR = 7.0            # SURVEY.md 8d contract figure
N_SM = 148

PAIR_WORKLOADS = {
    # name: (n, m, seed, pairs per step, description)
    "cfg1": (1000, 1000, 1, 10, "10 pairs 1000x1000, seed 1 (TestFile.cpp default: 10 tests), one call per pair"),
    "cfg2": (100000, 100000, 2, 1, "single pair 100000x100000, seed 2, MATCH=1 MISMATCH=-1 GAP_INIT=1 GAP_EXT=1"),
    "n1m": (1000000, 1000000, 6, 1, "single pair 1000000x1000000, seed 6"),
}
# one pair spread over the ring of all GPUs (strong scaling): boundary stream pushed GPU to GPU over NVLink
RING_WORKLOADS = {
    "ring400k": (400000, 400000, 7, "single pair 400000x400000, seed 7, DP bands cyclically striped over all GPUs"),
    "ring1m": (1000000, 1000000, 6, "single pair 1000000x1000000, seed 6, DP bands cyclically striped over all GPUs"),
    "cfg3": (4000000, 4000000, 3, "single pair 4000000x4000000, seed 3, DP bands cyclically striped over all GPUs"),
}
# batches of independent pairs, sharded pair-wise over the GPUs (no communication): (TOTAL pairs, len1, len2, seed, banded, text)
BATCH_WORKLOADS = {
    "cfg4": (10000000, 150, 1000, 4, False, "10M pairs, 150 bp reads vs 1 kb windows (half planted: 5% substitutions + 1% indels, half unrelated), pair-sharded"),
    "cfg4small": (400000, 150, 1000, 4, False, "400k pairs of the cfg4 recipe"),
    "cfg5": (1000000, 10000, 10000, 5, True, "1M pairs of 10 kb long reads (10% substitutions + 2% indels), band -32..31 (64 diagonals), pair-sharded"),
    "cfg5small": (40000, 10000, 10000, 5, True, "40k pairs of the cfg5 recipe"),
}
ALL_WORKLOADS = sorted(list(PAIR_WORKLOADS) + list(RING_WORKLOADS) + list(BATCH_WORKLOADS))


def golden_score(name):
    """Pinned scores: tests/golden/large_scores.json (oracle/gotoh_fast.c on the CPU: cfg2, ring400k, n1m, cfg3) and, for
    cfg2, the unmodified reference's own LazySmith (tests/golden/ref_scores_default.json)."""
    try:
        big = json.loads((ROOT / "tests" / "golden" / "large_scores.json").read_text())
        if name == "ring1m":
            name = "n1m"
        if name in big:
            return int(big[name]["score"])
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            while not self._halt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report that instead of inventing clocks
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def dump_outputs(args, env, name, values, dtype):
    """--dump-outputs: the scores of the last timed step of one record as DIR/<name>_scores[.rank<r>].npy."""
    if not args.dump_outputs:
        return
    out = np.asarray(values, dtype=dtype)
    if not np.array_equal(out, np.asarray(values)):
        raise SystemExit(f"bench.py: {name} scores are not exact in {np.dtype(dtype).name}")
    d = Path(args.dump_outputs)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{name}_scores{'' if env.world == 1 else f'.rank{env.rank}'}.npy", out)


def peak_gcups(f_mhz, vwidth, gpus=1):
    return gpus * N_SM * f_mhz * 1e6 * DPX_LANE_INSTR_PER_CLK_PER_SM * vwidth / INSTR_PER_CELL_VECTOR / 1e9


def cpu_reference_gcups(n_sample, seed, repeats=1):
    """Times the reference's own CPU path on a bounded sample of the workload; returns (gcups, kind, cores, text)."""
    import oracle_lib as O
    a = rng.random_acgt(seed, 0, n_sample)
    b = rng.random_acgt(seed, 1, n_sample)
    if O.ref_available():
        kind, fn = "reference", lambda: O.ref_call("ref_ParallelLazySmith_threads", a, b)
        what = "unmodified lazySmith_parallel_threads.cpp (ParallelLazySmith_threads, default args: sequential, lazySmith_parallel_threads.cpp:78-81)"
    else:
        kind, fn = "port", lambda: O.lazy_smith(a, b)
        what = "oracle port of LazySmith (oracle/_ref not present)"
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        s = fn()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return n_sample * n_sample / best / 1e9, kind, 1, f"{n_sample}x{n_sample} prefix of the workload pair, {what}; score {s}; host has {os.cpu_count()} cores"


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on this box's host cores.  Each step scores
    a bounded PREFIX of the workload pair (the reference needs ~54 s for the whole cfg2 pair; its rate is flat in N,
    SURVEY.md section 6), stated in config.sample; with --steps 1 the whole cfg2 pair is scored once."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload if args.workload in PAIR_WORKLOADS else "cfg2"
    n, m, seed, _, desc = PAIR_WORKLOADS[name]
    n_s = n if (args.steps == 1 and n <= 100000) else min(n, 8000)
    for _ in range(args.warmup):
        cpu_reference_gcups(2000, seed)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        g, kind, cores, text = cpu_reference_gcups(n_s, seed)
    dt = time.perf_counter() - t0
    value = n_s * n_s * args.steps / dt / 1e9
    sample = "the whole pair" if n_s == n else f"{n_s}x{n_s} prefix of the {n}x{m} pair per step (rate over rate: the reference's GCUPS is flat in N)"
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "GCUPS", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": name, "description": desc, "sample": sample, "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": round(value, 4), "unit": "GCUPS", "cores": cores, "kind": kind, "sample": text},
            "e2e": {"value": round(value, 4), "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def ncu_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the ncu --set full capture
    committed under profiles/ (only the bench default has one); None otherwise."""
    if workload != "cfg2":
        return None
    for name, key in (("r02_ncu_summary.json", "r02_cfg2_final.ncu-rep"), ("r01_ncu_summary.json", "r01_cfg2_final5.ncu-rep")):
        try:
            d = json.load(open(ROOT / "profiles" / name))
            return int(d[key]["dram_bytes_per_launch"])
        except Exception:
            continue
    return None


class Env:
    """torch / torch.distributed plumbing of one rank (device memory, streams, the barrier; not the product)."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from concurrentproject_b200 import api
        self.torch, self.dist, self.api = torch, dist, api
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.stream = torch.cuda.current_stream()

    def need_group(self):
        """The ring front end talks torch.distributed even on one GPU."""
        if not self.dist.is_initialized():
            s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
            self.dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                                         device_id=self.torch.device("cuda", self.local))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sum_over_ranks_i64(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.int64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [int(x) for x in t.tolist()]

    def close(self):
        if self.dist.is_initialized():
            self.dist.barrier()
            self.dist.destroy_process_group()


def pair_record(env, args, name):
    """One pair (cfg1: ten pairs) per GPU per step; rank r scores its own pair(s) (streams differ per rank): weak scaling."""
    torch, api = env.torch, env.api
    n, m, seed, pairs, desc = PAIR_WORKLOADS[name]
    import oracle_lib as O
    hosts = [(rng.random_acgt(seed, 2 * (env.rank * pairs + k), n), rng.random_acgt(seed, 2 * (env.rank * pairs + k) + 1, m)) for k in range(pairs)]
    devs = [(torch.from_numpy(a.copy()).cuda(), torch.from_numpy(b.copy()).cuda()) for a, b in hosts]
    if name == "cfg1":
        want = [O.gotoh_rolling(a, b) for a, b in hosts]              # every pair against the oracle
    else:
        want = [golden_score(name)] if env.rank == 0 else [None]
    ctx = api.Context(env.local)
    stream = env.stream
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def step_device():
        return [ctx.score_device(a.data_ptr(), n, b.data_ptr(), m, stream=stream.cuda_stream, no_linear=args.no_linear) for a, b in devs]

    def check(scores, what):
        for s, w in zip(scores, want):
            if w is not None and s != w:
                raise SystemExit(f"bench.py: {what} score {s} != pinned {w}")

    for _ in range(max(args.warmup, 3)):
        s = step_device()
    check(s, "device")
    env.barrier()
    sampler = ClockSampler(env.local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    engine_ms, launches, info = [], 0, {}
    for k in range(args.steps):
        flush.fill_(k & 0xFF)                      # L2 flush between timed steps (outside the event pair)
        ev[k][0].record(stream)
        s = step_device()
        ev[k][1].record(stream)
        info = ctx.last_run()
        engine_ms.append(info["engine_ms"])
        launches += pairs * (info["engine_launches"] + info["aux_launches"])
        check(s, "device")
    torch.cuda.synchronize()
    clocks = sampler.stop()
    dump_outputs(args, env, name, s, np.float64)
    dev_ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
    # end to end through the host-buffer call of the reference harness (TestFileWithGPU.cpp:92):
    # H2D of both sequences + encode + wavefront kernel + D2H of the result, wall clock per call
    for _ in range(2):
        [api.SmithWatermanScoreCUDA(a, b) for a, b in hosts]
    e2e_total = 0.0
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        s2 = [api.SmithWatermanScoreCUDA(a, b) for a, b in hosts]
        e2e_total += time.perf_counter() - t1
        check(s2, "e2e")
    dev_ms, e2e_ms = env.max_over_ranks([dev_ms, e2e_total * 1e3])
    cells = float(n) * float(m) * pairs
    value = cells * env.world * args.steps / (dev_ms * 1e-3) / 1e9
    e2e_val = cells * env.world * args.steps / (e2e_ms * 1e-3) / 1e9
    if env.rank != 0:
        return None
    k_ms = float(np.mean(engine_ms))
    f_mhz = clocks["sm_mhz"] or clocks["sm_max_mhz"] or 1965
    vwidth = 2 if info["lanes"] == 16 else 1
    peak = peak_gcups(f_mhz, vwidth)
    achieved = float(n) * float(m) / (k_ms * 1e-3) / 1e9
    cpu_g, kind, cores, text = cpu_reference_gcups(min(n, 12000), seed)
    return {
        "metric": METRIC, "value": round(value, 1), "unit": "GCUPS", "n_gpus": env.world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(dev_ms / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "s16x2" if info["lanes"] == 16 else "s32", "data": "synthetic",
        "config": {"workload": name, "description": desc, "pairs_per_gpu": pairs,
                   "l2": "flushed between timed steps (256 MiB write)", "kernel": info,
                   "score_checked_against": "oracle, every pair" if name == "cfg1" else ("pinned golden, every step" if want[0] is not None else None),
                   "score_checked_against_golden": want[0] is not None},
        "clocks": clocks,
        "e2e": {"value": round(e2e_val, 1), "unit": "GCUPS", "h2d_bytes_per_step": int(n + m) * pairs, "d2h_bytes_per_step": 40 * pairs,
                "call": "SmithWatermanScoreCUDA(host bytes) via libswb200.so C ABI, wall clock"},
        "gpu_launches": launches,
        "roofline": {"bound": "int_alu", "achieved": round(achieved, 1), "peak": round(peak, 1), "unit": "GCUPS",
                     "frac": round(achieved / peak, 4), "traffic": ncu_traffic(name),
                     "note": f"wavefront kernel only, {k_ms:.3f} ms/launch (CUDA events on its stream); traffic = DRAM bytes per launch "
                             f"from the committed ncu capture, algorithmic input is {(n + m) // 4} bytes, "
                             f"the boundary rows between CTAs stream through L2 (full-length links, partly written back); peak = 148 SM x {f_mhz} MHz x "
                             f"L={DPX_LANE_INSTR_PER_CLK_PER_SM:.0f} DPX lane-instr/clk/SM (measured, bench/intpeak.cu) x V={vwidth} / 7 "
                             "instr per cell vector (SURVEY.md 8d); not an HBM- or tensor-bound kernel"},
        "cpu_baseline": {"value": round(cpu_g, 4), "unit": "GCUPS", "cores": cores, "kind": kind, "sample": text},
    }


def ring_record(env, args, name, steps, warmup):
    """One long pair over all GPUs (strong scaling).  Every rank holds both sequences; the DP bands are dealt
    cyclically to the warps of all GPUs and the boundary stream crosses GPUs inside the kernel."""
    torch, dist = env.torch, env.dist
    from concurrentproject_b200.ring import DistributedRingAligner
    env.need_group()
    n, m, seed, desc = RING_WORKLOADS[name]
    want = golden_score(name)
    a_h = rng.random_acgt(seed, 0, n)
    b_h = rng.random_acgt(seed, 1, m)
    a_d = torch.from_numpy(a_h.copy()).cuda()
    b_d = torch.from_numpy(b_h.copy()).cuda()
    al = DistributedRingAligner(env.local, min(n, m))
    stream = env.stream
    lanes = 32 if args.lanes32 else 0             # default: library policy (re-based 16-bit lanes for long pairs)
    two_sided = -1 if args.one_sided else 0
    scores = []
    for _ in range(max(warmup, 1)):
        scores.append(al.score(a_d.data_ptr(), n, b_d.data_ptr(), m, lanes=lanes, stream=stream.cuda_stream, two_sided=two_sided))
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(env.local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    kms = []
    for _ in range(steps):
        scores.append(al.score(a_d.data_ptr(), n, b_d.data_ptr(), m, lanes=lanes, stream=stream.cuda_stream, two_sided=two_sided))
        kms.append(al.last_run()["engine_ms"])
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    dump_outputs(args, env, name, [scores[-1]], np.float64)
    # end to end: every step copies both sequences from pinned host memory and reads the score back
    a_p, b_p = torch.from_numpy(a_h.copy()).pin_memory(), torch.from_numpy(b_h.copy()).pin_memory()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        a_d.copy_(a_p, non_blocking=True)
        b_d.copy_(b_p, non_blocking=True)
        scores.append(al.score(a_d.data_ptr(), n, b_d.data_ptr(), m, lanes=lanes, stream=stream.cuda_stream, two_sided=two_sided))
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    ms, e2e_ms, k_ms = env.max_over_ranks([e0.elapsed_time(e1), e2e_ms, float(np.mean(kms))])
    if len(set(scores)) != 1:
        raise SystemExit(f"bench.py: ring scores differ between steps: {scores}")
    if want is not None and scores[-1] != want:
        raise SystemExit(f"bench.py: ring score {scores[-1]} != pinned {want}")
    info = al.last_run()
    al.close()
    if env.rank != 0:
        return None
    cells = float(n) * float(m)
    value = cells * steps / (ms * 1e-3) / 1e9
    f_mhz = clocks["sm_mhz"] or 1965
    vwidth = 2 if info["lanes"] == 16 else 1
    peak = peak_gcups(f_mhz, vwidth, env.world)
    return {"metric": METRIC, "value": round(value, 1), "unit": "GCUPS", "n_gpus": env.world, "steps": steps,
            "warmup": max(warmup, 1), "ms_per_step": round(ms / steps, 3), "kernel_ms_max_over_ranks": round(k_ms, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": ("s16x2 re-based" if info.get("rebased") else "s16x2") if info["lanes"] == 16 else "s32", "data": "synthetic",
            "config": {"workload": name, "description": desc, "l2": "working set is registers; boundary rings stream through L2",
                       "kernel": info, "score": scores[-1], "score_checked_against_golden": want is not None},
            "clocks": clocks, "gpu_launches": (info["engine_launches"] + info["aux_launches"]) * steps,
            "e2e": {"value": round(cells * steps / (e2e_ms * 1e-3) / 1e9, 1), "unit": "GCUPS",
                    "h2d_bytes_per_step": int(n + m) * env.world, "d2h_bytes_per_step": 16 * env.world,
                    "call": "DistributedRingAligner.score after copying both sequences from pinned host memory on every rank, wall clock, max over ranks"},
            "roofline": {"bound": "int_alu", "achieved": round(value, 1), "peak": round(peak, 1), "unit": "GCUPS",
                         "frac": round(value / peak, 4), "traffic": None,
                         "note": f"whole ring of {env.world} GPU(s); peak = {env.world} x 148 SM x {f_mhz} MHz x L=64 x V={vwidth} / 7"}}


def batch_record(env, args, name, steps, warmup):
    """A fixed total batch cut into contiguous ranges of pairs, one per GPU (strong scaling, no communication on the
    data path).  Inputs come from the seeded device generator by GLOBAL pair id, so every GPU count scores the very
    same pairs; a sample is regenerated on the host (rng.read_pair / rng.long_pair) and checked against the oracle."""
    torch, api = env.torch, env.api
    import oracle_lib as O
    total, l1, l2, seed, banded, desc = BATCH_WORKLOADS[name]
    per = (total + env.world - 1) // env.world
    k0 = min(total, env.rank * per)
    npairs = min(total, k0 + per) - k0
    stream = env.stream
    seq1 = torch.empty((max(npairs, 1), l1), dtype=torch.uint8, device="cuda")
    seq2 = torch.empty((max(npairs, 1), l2), dtype=torch.uint8, device="cuda")
    if banded:
        api.gen_long_pairs_device(env.local, seed, k0, npairs, l1, seq1.data_ptr(), seq2.data_ptr(), stream.cuda_stream)
    else:
        api.gen_read_pairs_device(env.local, seed, k0, npairs, l1, l2, seq1.data_ptr(), seq2.data_ptr(), stream.cuda_stream)
    off1 = (torch.arange(npairs, device="cuda", dtype=torch.int64) * l1).contiguous()
    off2 = (torch.arange(npairs, device="cuda", dtype=torch.int64) * l2).contiguous()
    len1 = torch.full((npairs,), l1, dtype=torch.int32, device="cuda")
    len2 = torch.full((npairs,), l2, dtype=torch.int32, device="cuda")
    scores = torch.zeros(npairs, dtype=torch.int32, device="cuda")
    ctx = api.Context(env.local)
    lo, hi = -32, 31
    if banded:     # exact in-band cell count of one n x m pair (i = row in seq2, j = column in seq1)
        i = np.arange(1, l2 + 1)
        per_pair = int(np.maximum(0, np.minimum(l1, i + hi) - np.maximum(1, i + lo) + 1).sum())
    else:
        per_pair = l1 * l2
    cells_total = float(total) * per_pair
    batch = api.PackedBatch(ctx, seq1.data_ptr(), off1.data_ptr(), len1.data_ptr(), seq2.data_ptr(), off2.data_ptr(),
                            len2.data_ptr(), npairs, l1, l2, int(float(npairs) * per_pair), stream=stream.cuda_stream, keep_order=banded)

    def run_kernel():
        if banded:
            batch.score_banded(scores.data_ptr(), lo, hi, stream=stream.cuda_stream, no_linear=args.no_linear, config=args.banded_config)
        else:
            batch.score(scores.data_ptr(), stream=stream.cuda_stream, no_linear=args.no_linear)

    for _ in range(max(warmup, 3)):
        run_kernel()
    # parity on a seeded sample of pairs, regenerated on the HOST from their global ids, against the oracle
    want_sample = (1000 if banded else 10000) // env.world
    idx = np.unique(np.linspace(0, max(npairs - 1, 0), num=min(want_sample, npairs)).astype(np.int64)) if npairs else np.zeros(0, dtype=np.int64)
    gen = (lambda k: rng.long_pair(seed, k, l1)) if banded else (lambda k: rng.read_pair(seed, k, l1, l2))
    hp = [gen(int(k0 + p)) for p in idx]
    got = scores[torch.from_numpy(idx).cuda()].cpu().numpy() if len(idx) else np.zeros(0, dtype=np.int32)
    if len(idx):
        want = O.gotoh_banded_batch([a for a, _ in hp], [b for _, b in hp], lo, hi) if banded else O.gotoh_batch([a for a, _ in hp], [b for _, b in hp])
        if want.tolist() != got.tolist():
            bad = int(np.argmax(want != got))
            raise SystemExit(f"bench.py: batch scores differ from the oracle on the sample (pair {int(k0 + idx[bad])}: {int(got[bad])} != {int(want[bad])})")

    def checksum():   # 64-bit, position dependent, over ALL scores of this rank (global pair ids)
        ids = torch.arange(k0, k0 + npairs, device="cuda", dtype=torch.int64)
        s64 = scores.to(torch.int64)
        return int(s64.sum()), int((s64 * (ids % 1000003 + 1)).sum())       # < 2^63 for every workload here

    chk = checksum()
    env.barrier()
    sampler = ClockSampler(env.local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    kms = []
    for _ in range(steps):      # packed inputs per pass are far larger than L2: no flush needed
        run_kernel()
        kms.append(ctx.last_run()["engine_ms"])
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    dev_ms = e0.elapsed_time(e1)
    if checksum() != chk:
        raise SystemExit("bench.py: batch checksum changed between passes")
    dump_outputs(args, env, name, scores.cpu().numpy(), np.float32)    # cfg4: 10 M pairs, 40 MB
    # end to end from HOST bytes: H2D of the sequences, pack, kernel, D2H of the scores, through the C ABI host call
    ne = min(npairs, 2500000 if not banded else 250000)
    r_e, w_e = seq1[:ne].cpu().pin_memory().numpy().reshape(-1), seq2[:ne].cpu().pin_memory().numpy().reshape(-1)
    o1, o2 = off1[:ne].cpu().pin_memory().numpy(), off2[:ne].cpu().pin_memory().numpy()
    ln1, ln2 = len1[:ne].cpu().pin_memory().numpy(), len2[:ne].cpu().pin_memory().numpy()
    del seq1, seq2
    torch.cuda.empty_cache()

    def host_call():
        if banded:
            return api.score_banded_batch_flat(r_e, o1, ln1, w_e, o2, ln2, lo, hi)
        return api.score_batch_flat(r_e, o1, ln1, w_e, o2, ln2)

    out = host_call() if ne else np.zeros(0, dtype=np.int32)
    env.barrier()
    t1 = time.perf_counter()
    for _ in range(steps):
        out = host_call() if ne else out
    e2e_s = (time.perf_counter() - t1) / steps      # per call
    if out.tolist() != scores[:ne].cpu().numpy().tolist():
        raise SystemExit("bench.py: host batch call disagrees with the device-resident pass")
    # the same call with the host batch already in the resident 2-bit format (a quarter of the PCIe bytes, no pack kernel)
    e2e_packed_s, np_pk = 0.0, 0
    if ne:
        np_pk = min(ne, 1000000)
        pin = lambda x: torch.from_numpy(x).pin_memory().numpy()
        if banded:
            w1, st1, w2, st2 = api.pack_banded_host(r_e[:np_pk * l1], o1[:np_pk], ln1[:np_pk], w_e[:np_pk * l2], o2[:np_pk], ln2[:np_pk])
            w1, w2 = pin(w1), pin(w2)
            packed_call = lambda: api.score_banded_batch_packed(w1, st1, w2, st2, ln1[:np_pk], ln2[:np_pk], lo, hi)
        else:
            qw, qs, tw, ts, ql, tl = api.pack_batch_host(r_e[:np_pk * l1], o1[:np_pk], ln1[:np_pk], w_e[:np_pk * l2], o2[:np_pk], ln2[:np_pk])
            qw, tw, ql, tl = pin(qw), pin(tw), pin(ql), pin(tl)
            packed_call = lambda: api.score_batch_packed(qw, qs, tw, ts, ql, tl)
        packed_call()
        env.barrier()
        t1 = time.perf_counter()
        for _ in range(steps):
            outp = packed_call()
        e2e_packed_s = (time.perf_counter() - t1) / steps      # per call
        if outp.tolist() != out[:np_pk].tolist():
            raise SystemExit("bench.py: packed host batch call disagrees with the byte call")
    dev_ms, e2e_ms, k_ms, e2e_packed_ms = env.max_over_ranks([dev_ms, e2e_s * 1e3, float(np.mean(kms)), e2e_packed_s * 1e3])
    sum_scores, weighted, n_checked, ne_total, np_pk_total = env.sum_over_ranks_i64([chk[0], chk[1], len(idx), ne, np_pk])
    info = ctx.last_run()
    batch.close()
    if env.rank != 0:
        return None
    value = cells_total * steps / (dev_ms * 1e-3) / 1e9
    e2e_val = float(ne_total) * per_pair / (e2e_ms * 1e-3) / 1e9
    f_mhz = clocks["sm_mhz"] or 1965
    peak = peak_gcups(f_mhz, 2, env.world)
    # reference CPU on a sample: one reference call per pair, spread over the host cores
    rs, ws = [a for a, _ in hp][:500 if banded else 4000], [b for _, b in hp][:500 if banded else 4000]
    t0 = time.perf_counter()
    if banded:
        cores, kind = O.oracle().oracle_max_threads(), "port"
        O.gotoh_banded_batch(rs, ws, lo, hi)
    elif O.ref_available():
        import ctypes as C
        f1, o1s, l1s = O._batch_args(rs)
        f2, o2s, l2s = O._batch_args(ws)
        outb = np.zeros(len(rs), dtype=np.int32)
        cores, kind = os.cpu_count() or 1, "reference"
        O.ref().ref_batch(2, O._ptr(f1), o1s.ctypes.data_as(C.POINTER(C.c_longlong)), l1s.ctypes.data_as(C.POINTER(C.c_int)),
                          O._ptr(f2), o2s.ctypes.data_as(C.POINTER(C.c_longlong)), l2s.ctypes.data_as(C.POINTER(C.c_int)),
                          len(rs), cores, outb.ctypes.data_as(C.POINTER(C.c_int)))
    else:
        cores, kind = O.oracle().oracle_max_threads(), "port"
        O.gotoh_batch(rs, ws)
    cpu_g = len(rs) * per_pair / (time.perf_counter() - t0) / 1e9
    return {"metric": METRIC, "value": round(value, 1), "unit": "GCUPS", "n_gpus": env.world, "steps": steps,
            "warmup": max(warmup, 3), "ms_per_step": round(dev_ms / steps, 3), "kernel_ms_max_over_ranks": round(k_ms, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "s16x2",
            "data": "synthetic (seeded device generator, csrc/swb_gen.cu = concurrentproject_b200/rng.py)",
            "config": {"workload": name, "description": desc, "pairs_total": total, "pairs_per_gpu": per,
                       "l2": "packed inputs per pass are far larger than L2", "kernel": info,
                       "sample_checked_against_oracle": n_checked,
                       "checksum": {"sum_of_scores": sum_scores, "weighted": weighted,
                                    "note": "over ALL pairs, by global pair id: identical for every GPU count"}},
            "clocks": clocks, "gpu_launches": steps,
            "e2e": {"value": round(e2e_val, 1), "unit": "GCUPS", "h2d_bytes_per_step": int(ne * (l1 + l2 + 24)) * env.world,
                    "d2h_bytes_per_step": int(4 * ne) * env.world,
                    "call": f"swb200_score{'_banded' if banded else ''}_batch(pinned host bytes) on {ne} pairs per GPU ({ne_total} in all), wall clock, max over ranks"},
            "e2e_packed": None if not np_pk_total else {
                "value": round(float(np_pk_total) * per_pair / (e2e_packed_ms * 1e-3) / 1e9, 1), "unit": "GCUPS",
                "h2d_bytes_per_step": int(np_pk * ((l1 + 31) // 32 + (l2 + 31) // 32 + (4 if banded else 2)) * 8 + np_pk * 8) * env.world, "d2h_bytes_per_step": int(4 * np_pk) * env.world,
                "call": f"swb200_score{'_banded' if banded else ''}_batch_packed(pinned host words, 2 bits per base) on {np_pk} pairs per GPU, wall clock, max over ranks"},
            "roofline": {"bound": "int_alu", "achieved": round(value, 1), "peak": round(peak, 1), "unit": "GCUPS",
                         "frac": round(value / peak, 4), "traffic": None,
                         "note": f"batch kernel on {env.world} GPU(s); peak = {env.world} x 148 SM x {f_mhz} MHz x L=64 x V=2 / 7"},
            "cpu_baseline": {"value": round(cpu_g, 3), "unit": "GCUPS", "cores": cores, "kind": kind,
                             "sample": (f"{len(rs)} pairs of the batch, oracle_gotoh_banded per pair over {cores} threads (the reference has no banded mode)"
                                        if banded else
                                        f"{len(rs)} pairs of the batch, one ParallelLazySmith_threads call per pair, pairs spread over {cores} host threads")}}


def run_ours(args):
    env = Env()
    name = args.workload
    if name in RING_WORKLOADS:
        line = ring_record(env, args, name, args.steps, args.warmup)
    elif name in BATCH_WORKLOADS:
        line = batch_record(env, args, name, args.steps, args.warmup)
    else:
        line = pair_record(env, args, name)
        if name == "cfg2" and not args.no_extra:
            # the two multi-GPU designs of BASELINE configs 3 and 4 on the same N GPUs, in the same run
            ring = ring_record(env, args, "cfg3", args.steps, args.warmup)
            batch = batch_record(env, args, "cfg4", args.steps, args.warmup)
            if env.rank == 0:
                line["ring"] = ring
                line["batch"] = batch
    if env.rank == 0:
        print(json.dumps(line), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=ALL_WORKLOADS)
    ap.add_argument("--no-extra", action="store_true", help="headline only: skip the cfg3 ring and cfg4 batch sub-records")
    ap.add_argument("--lanes32", action="store_true", help="ring workloads: force the 32-bit kernel")
    ap.add_argument("--banded-config", type=int, default=0, help="banded workloads: 0 = 4 threads per pair (default), 2 / 8 / 16 = the other kernel layouts")
    ap.add_argument("--one-sided", action="store_true", help="ring workloads: never sweep from both ends")
    ap.add_argument("--no-linear", action="store_true",
                    help="keep the general affine kernel although GAP_INIT == GAP_EXT (default: use the exact E/F-free kernel)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the scores the timed path returned in its last step as DIR/<workload>_scores.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has nothing to dump")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
