"""Drop-in proof: the reference's own, unmodified TestFileWithGPU.cpp linked against libswb200.so instead of
simpleGPU.cu / cudaLazy.cu / cudaSmithM.cu (oracle/Makefile `dropin`, built where /root/reference exists; the
binary travels to the GPU box in the git-ignored oracle/_ref/).  Its success predicate compares the three
reference CPU functions with our three GPU functions on 10 random 3000x3000 pairs (TestFileWithGPU.cpp:105)."""
import json
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu


def _run(exe, stdin=None, args=()):
    return subprocess.run([str(exe), *args], input=stdin, capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_unmodified_reference_harness_links_and_agrees():
    exe = ROOT / "oracle" / "_ref" / "test_runner2"
    if not exe.exists():
        pytest.skip("oracle/_ref/test_runner2 not built (needs /root/reference at build time)")
    out = _run(exe, stdin="1\n")                       # mode 1: per-test lines (TestFileWithGPU.cpp:176-183)
    assert out.returncode == 0, out.stderr
    assert out.stdout.count("SUCCESS") == 10 and "ERROR" not in out.stdout, out.stdout[-2000:]
    out = _run(exe, stdin="2\n")                       # mode 2: averages
    assert "Success: 1" in out.stdout and "ERROR" not in out.stdout


def test_own_harness_with_reference_cpu_functions():
    """The harness's GPU functions against the reference's three CPU functions on the same seeded pairs: linked in
    (oracle/Makefile `harness_ref`) when built, and through the reference's stored scores when they are committed."""
    exe = ROOT / "oracle" / "_ref" / "test_runner_b200_ref"
    live = ROOT / "tests" / "golden" / "ref_scores_live.json"
    if not exe.exists() and not live.exists():
        pytest.skip("needs the original project: oracle/_ref/test_runner_b200_ref or tests/golden/ref_scores_live.json "
                    "(written by tests/golden/make_golden.py --live)")
    if exe.exists():
        out = _run(exe, args=("2", "8", "1", "50", "500", "1000", "3000"))
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr
        assert out.stdout.count("Success: 1") == 5
    if live.exists():
        h = json.loads(live.read_text())["harness"]
        assert all(three == [three[0]] * 3 for three in h["scores"])
        runner = ROOT / "harness" / "test_runner_b200"
        if not runner.exists():
            subprocess.run(["make", "-s", "-C", str(ROOT / "harness")], check=True)
        out = _run(runner, args=("1", str(h["seed"]), *map(str, h["lengths"])))   # mode 1: one line per pair
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr
        got = [int(s) for s in re.findall(r"^TEST \d+: score=(-?\d+) SUCCESS", out.stdout, re.M)]
        assert got == [three[0] for three in h["scores"]]


def test_own_harness_gpu_only():
    exe = ROOT / "harness" / "test_runner_b200"
    if not exe.exists():
        subprocess.run(["make", "-s", "-C", str(ROOT / "harness")], check=True)
    out = _run(exe, args=("1", "8", "100", "2000"))
    assert out.returncode == 0 and out.stdout.count("SUCCESS") == 20, out.stdout[-2000:]
