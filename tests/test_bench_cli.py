"""bench.py's contract that can be checked without a GPU: the command line parses, and the reference arm
(`--impl reference`: the reference's own dual_func from oracle/_ref on the host cores, or the oracle port of it where the
reference was not built) prints ONE JSON line -- same metric / unit / config vocabulary as the GPU arm, `impl`,
`cpu_baseline` and an `e2e` block that repeats the line's own value with zero transfer bytes."""
import json
import os
import subprocess
import sys

import pytest

import oracle_bindings as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_help_parses():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--gpus" in r.stdout and "--impl" in r.stdout and "--steps" in r.stdout


@pytest.mark.parametrize("alg", ["ccsaq", "mma"])
def test_reference_arm_prints_the_contract_line(alg):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--n", "100000", "--alg", alg], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ccsa_dual_evals_per_sec" and d["unit"] == "dual-evals/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] - 1.0) < 0.2       # one dual evaluation per step
    assert d["config"]["n"] == 100000 and d["config"]["m"] == 4
    assert d["cpu_baseline"]["kind"] == ("reference" if ob.ref_dual_available() else "port") and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
