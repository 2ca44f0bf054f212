"""bench.py contract checks.  Without a GPU: the reference arm (--impl reference) runs the unmodified reference
CPU function (oracle/_ref/libref.so, or the oracle port where the reference sources are absent) and prints one
JSON line with the keys a caller reads, and bad step counts are refused.  On a GPU: --dump-outputs writes the
scores of the last timed step."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    # two steps: each scores a bounded prefix of the pair (one step would score the whole 100 000 x 100 000 pair, ~1-2 min)
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GCUPS" and line["higher_is_better"] is True
    assert line["config"]["workload"] == "cfg2" and line["n_gpus"] == 1 and line["steps"] == 2
    assert "prefix" in line["config"]["sample"]          # the line says that a step is a sample of the workload, and which
    assert line["value"] > 0 and abs(line["value"] - line["e2e"]["value"]) < 1e-9
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"]


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_scores_of_the_last_step(tmp_path):
    import numpy as np
    import oracle_lib as O
    from concurrentproject_b200 import rng
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "cfg1", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    kernel = line["config"]["kernel"]        # launches are counted inside the timed loop: 2 steps x 10 pairs
    assert line["steps"] == 2 and line["gpu_launches"] == 2 * 10 * (kernel["engine_launches"] + kernel["aux_launches"]) > 0
    assert [p.name for p in tmp_path.iterdir()] == ["cfg1_scores.npy"]
    got = np.load(tmp_path / "cfg1_scores.npy")
    want = [O.gotoh_rolling(rng.random_acgt(1, 2 * k, 1000), rng.random_acgt(1, 2 * k + 1, 1000)) for k in range(10)]
    assert got.dtype == np.float64 and got.tolist() == want


def test_workload_table_names_the_baseline_configs():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    base = json.load(open(ROOT / "BASELINE.json"))
    assert b.METRIC and "GCUPS" in b.METRIC
    for k in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
        assert k in b.PAIR_WORKLOADS or k in b.RING_WORKLOADS or k in b.BATCH_WORKLOADS, k
    for name in ("cfg2", "n1m", "cfg3"):                 # every long pair the bench scores has a pinned score
        assert b.golden_score(name), name
    assert b.golden_score("cfg3") == 456968
    assert "metric" in base
