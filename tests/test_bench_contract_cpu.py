"""bench.py's reference arm (the unmodified reference from oracle/_ref on the host cores; the oracle port
when that install is absent) keeps the JSON contract the driver reads:
one line, the same metric / unit as our arm, a cpu_baseline describing the run and a zero-copy e2e object."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference"
    assert j["metric"].startswith("DREAM chain-steps/s") and j["unit"] == "chain-steps/s"
    assert j["higher_is_better"] is True and j["scaling"] == "weak" and j["vs_baseline"] is None
    assert j["dtype"] == "f64" and j["data"] == "synthetic" and j["steps"] == 2 and j["n_gpus"] == 1
    assert j["value"] > 0 and j["ms_per_step"] > 0
    assert "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    sys.path.insert(0, ROOT)
    from oracle import ref_runner
    have_ref = ref_runner.reference_dir() is not None
    assert cb["kind"] == ("reference" if have_ref else "port")
    assert cb["cores"] >= 1 and cb["value"] == j["value"] and cb["sample"]
    e = j["e2e"]
    assert e["value"] == j["value"] and e["unit"] == j["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.parametrize("args", [["--steps", "0"], ["--gpus", "2", "--dump-outputs", "x"],
                                  ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_refuses_bad_arguments(args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 2 and "error:" in r.stderr


def test_reference_runner_shared_memory_ranks():
    """oracle/ref_runner.py: the unmodified reference on 2 shared-memory ranks grows every chain by exactly
    one state per generation (demc.py:79-135) -- the step count the baseline divides by."""
    import pytest
    sys.path.insert(0, ROOT)
    from oracle import ref_runner
    if ref_runner.reference_dir() is None:
        pytest.skip("the unmodified reference is not installed in oracle/_ref")
    spec = dict(n_chains=8, dim=100, algo="dream", seed=42, ctor_kwargs=dict(n_cr_gen=2, burnin_gen=100))
    dt, steps = ref_runner.time_reference(spec, 2, gens=3, gens_warm=1)
    assert steps == 8 * 3 and dt > 0
