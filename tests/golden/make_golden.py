#!/usr/bin/env python
"""Generates the committed fixtures under tests/golden/ by running the UNMODIFIED reference.

Run in the build container (needs /root/reference and g++):   python tests/golden/make_golden.py
It (1) builds oracle/_ref/libref.so from the reference sources where they lie, (2) regenerates the
reference's seeded inputs (cudaSmithM.cu:200-213) with gen_mt_pairs.cpp and checks the scores the
reference itself records (cudaSmithM.cu:285-294, 314-323, 342-351), (3) scores mix64-generated pairs
with the reference's three CPU functions, (4) does the same with the reference's constants replaced
(sed copy in /tmp, oracle/Makefile ref_params) for the non-default parameter sets of SURVEY.md 8c.
Nothing here is imported by the product; the GPU box only ever sees the written fixtures.
"""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import oracle_lib as O  # noqa: E402
from concurrentproject_b200 import rng  # noqa: E402

REF = Path("/root/reference")
RECORDED = {  # cudaSmithM.cu:285-294, 314-323, 342-351
    32: [6, 16, 5, 6, 5, 6, 6, 8, 8, 5],
    516: [65, 56, 56, 72, 69, 61, 70, 62, 56, 56],
    4096: [466, 472, 474, 497, 486, 442, 454, 478, 451, 471],
}


def main(big: bool):
    assert REF.is_dir(), "needs /root/reference"
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), "all", "ref"], check=True)

    # (2) the reference's own seeded inputs ---------------------------------------------------
    exe = Path("/tmp/swb200_gen_mt_pairs")
    subprocess.run(["/usr/bin/g++", "-O2", "-o", str(exe), str(HERE / "gen_mt_pairs.cpp")], check=True)
    for L, want in RECORDED.items():
        out = subprocess.run([str(exe), str(L)], check=True, capture_output=True, text=True).stdout.split("\n")
        lines = []
        for k, line in enumerate(l for l in out if l):
            a, b = line.split()
            s_main = O.ref_call("ref_SmithWatermanScore", a, b)
            s_lazy = O.ref_call("ref_LazySmith", a, b)
            s_thr = O.ref_call("ref_ParallelLazySmith_threads", a, b)
            assert s_main == s_lazy == s_thr == want[k], (L, k, s_main, s_lazy, s_thr, want[k])
            lines.append(f"{a} {b} {s_main}")
        (HERE / f"mt12345_L{L}.txt").write_text("\n".join(lines) + "\n")
        print(f"mt12345 L={L}: reference reproduces its recorded scores {want}")

    # (3) mix64 pairs scored by the reference, default parameters ------------------------------
    cases = []
    shapes = [(0, 0), (0, 7), (5, 0), (1, 1), (1, 9), (2, 2), (3, 5), (17, 4), (31, 33), (64, 64), (65, 63),
              (100, 100), (127, 129), (128, 128), (150, 1000), (1000, 150), (255, 257), (333, 777), (512, 512),
              (1000, 1000), (1000, 1000), (1000, 1000), (1023, 2049), (2048, 1024), (3000, 3000), (2500, 4100)]
    for k, (n, m) in enumerate(shapes):
        a = rng.random_acgt(1, 2 * k, n)
        b = rng.random_acgt(1, 2 * k + 1, m)
        s_main = O.ref_call("ref_SmithWatermanScore", a, b)
        s_lazy = O.ref_call("ref_LazySmith", a, b)
        s_thr = O.ref_call("ref_ParallelLazySmith_threads", a, b)
        assert s_main == s_lazy == s_thr
        cases.append({"kind": "random", "seed": 1, "stream1": 2 * k, "stream2": 2 * k + 1, "n": n, "m": m, "score": s_main})
    # planted similarity: seq2 = mutate(seq1)
    for k, (n, sub, indel) in enumerate([(200, 0.05, 0.01), (1000, 0.05, 0.01), (1000, 0.10, 0.02), (2000, 0.02, 0.0),
                                         (3000, 0.10, 0.02), (1500, 0.0, 0.05), (800, 0.3, 0.1)]):
        a = rng.random_acgt(7, k, n)
        b = rng.mutate(a, 7, 1000 + k, sub, indel)
        s_main = O.ref_call("ref_SmithWatermanScore", a, b)
        s_lazy = O.ref_call("ref_LazySmith", a, b)
        assert s_main == s_lazy
        cases.append({"kind": "planted", "seed": 7, "stream1": k, "mut_stream": 1000 + k, "n": n, "m": int(len(b)),
                      "sub": sub, "indel": indel, "score": s_main})
    # longer, rolling-row reference only (main.cpp needs 12*n*m bytes)
    for k, n in enumerate([8000, 20000]):
        a = rng.random_acgt(3, 2 * k, n)
        b = rng.random_acgt(3, 2 * k + 1, n)
        s_lazy = O.ref_call("ref_LazySmith", a, b)
        s_thr = O.ref_call("ref_ParallelLazySmith_threads", a, b)
        assert s_lazy == s_thr
        cases.append({"kind": "random", "seed": 3, "stream1": 2 * k, "stream2": 2 * k + 1, "n": n, "m": n, "score": s_lazy,
                      "by": "LazySmith"})
    if big:
        # BASELINE cfg2: one 100 000 x 100 000 pair, seed 2 (reference LazySmith: ~100 s)
        n = 100000
        a = rng.random_acgt(2, 0, n)
        b = rng.random_acgt(2, 1, n)
        s_lazy = O.ref_call("ref_LazySmith", a, b)
        cases.append({"kind": "random", "seed": 2, "stream1": 0, "stream2": 1, "n": n, "m": n, "score": s_lazy,
                      "by": "LazySmith", "config": "cfg2"})
    else:
        old = json.loads((HERE / "ref_scores_default.json").read_text()) if (HERE / "ref_scores_default.json").exists() else []
        cases += [c for c in old if c.get("config") == "cfg2"]
    (HERE / "ref_scores_default.json").write_text(json.dumps(cases, indent=0) + "\n")
    print(f"default-parameter fixtures: {len(cases)} cases")

    # (4) non-default constants (match, mismatch, gap_init, gap_ext) ----------------------------
    psets = [(2, -3, 5, 1), (5, -4, 11, 1), (2, -1, 2, 1), (2, -1, 3, 1), (5, -4, 6, 2), (1, -1, 4, 2), (3, -2, 2, 2), (1, -3, 1, 1)]
    pcases = []
    for p in psets:
        ma, mi, gi, ge = p
        subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), "ref_params", f"GI={gi}", f"GE={ge}", f"MA={ma}", f"MI={mi}"],
                       check=True, capture_output=True)
        for k in range(12):
            n = [50, 200, 333, 700, 1000, 1200, 150, 64, 1, 400, 900, 1500][k]
            m = [60, 180, 777, 700, 1000, 500, 1000, 64, 5, 401, 300, 1500][k]
            a = rng.random_acgt(11, 2 * k, n)
            if k % 3 == 0:
                b = rng.mutate(a, 11, 500 + k, 0.08, 0.04)
            else:
                b = rng.random_acgt(11, 2 * k + 1, m)
            s_main = O.ref_call("ref_SmithWatermanScore", a, b, p)
            s_lazy = O.ref_call("ref_LazySmith", a, b, p)
            pcases.append({"params": list(p), "seed": 11, "stream1": 2 * k, "stream2": 2 * k + 1, "mut_stream": 500 + k,
                           "planted": k % 3 == 0, "n": n, "m": int(len(b)), "score_main": s_main, "score_lazy": s_lazy})
    (HERE / "ref_scores_params.json").write_text(json.dumps(pcases, indent=0) + "\n")
    ndiff = sum(c["score_main"] != c["score_lazy"] for c in pcases)
    print(f"parameterised fixtures: {len(pcases)} cases, lazy != main in {ndiff}")


def fresh_inputs():
    """The 25 seeded pairs of tests/test_oracle.py::test_oracle_equals_live_reference_on_fresh_inputs."""
    for k in range(25):
        n, m = 1 + int(rng.mix64(41, 1, k) % 700), 1 + int(rng.mix64(41, 2, k) % 700)
        a, b = rng.random_acgt(41, 2 * k, n), rng.random_acgt(41, 2 * k + 1, m)
        if k % 4 == 0:
            b = rng.mutate(a, 41, 900 + k, 0.07, 0.03)
        yield a, b


HARNESS_SEED, HARNESS_LENGTHS, HARNESS_TESTS = 8, (1, 50, 500, 1000, 3000), 10


def harness_inputs():
    """The pairs harness/test_runner_b200 scores with seed 8 at these lengths (its random_sequence = rng.random_acgt)."""
    for n in HARNESS_LENGTHS:
        for it in range(HARNESS_TESTS):
            yield rng.random_acgt(HARNESS_SEED, 2 * it, n), rng.random_acgt(HARNESS_SEED, 2 * it + 1, n)


def live():
    """(5) ref_scores_live.json: the scores of the reference's three CPU functions (SmithWatermanScore, LazySmith,
    ParallelLazySmith_threads) on the inputs that tests/test_oracle.py and tests/test_gpu_dropin.py otherwise compare
    with the reference live.  Needs oracle/_ref/libref.so."""
    assert O.ref_available(), "needs oracle/_ref/libref.so"
    fns = ("ref_SmithWatermanScore", "ref_LazySmith", "ref_ParallelLazySmith_threads")
    out = {"functions": list(fns),
           "fresh": [[O.ref_call(f, a, b) for f in fns] for a, b in fresh_inputs()],
           "harness": {"seed": HARNESS_SEED, "lengths": list(HARNESS_LENGTHS), "tests": HARNESS_TESTS,
                       "scores": [[O.ref_call(f, a, b) for f in fns] for a, b in harness_inputs()]}}
    (HERE / "ref_scores_live.json").write_text(json.dumps(out) + "\n")
    print(f"live-comparison fixtures: {len(out['fresh'])} fresh pairs, {len(out['harness']['scores'])} harness pairs")


if __name__ == "__main__":
    if "--live" in sys.argv:
        live()
    else:
        main(big="--big" in sys.argv)
