"""bench.py --dump-outputs: the timed generations' results land in DIR as float64 .npy files within 64 MB, the
same arguments give the same files, and --steps is the number of timed generations."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)


@pytest.mark.gpu
def test_dump_outputs_are_complete_and_repeatable(tmp_path):
    runs = []
    for i in range(2):
        d = tmp_path / ("run%d" % i)
        r = _bench("--gpus", "1", "--steps", "4", "--warmup", "3", "--no-cpu", "--no-e2e", "--no-stationary",
                   "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 4
        runs.append(dict((f[:-4], np.load(str(d / f))) for f in sorted(os.listdir(str(d)))))
    a, b = runs
    assert sorted(a) == ["accepted_rejected", "delta_m", "history_sample", "lnl", "p_cr", "state_sample",
                         "state_sample_rows"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["state_sample"].shape == (8192, 100) and a["lnl"].shape == (100000,)
    # the history rows of the 4 timed generations; the newest, left pending by the fused kernel, is the state
    assert a["history_sample"].shape == (4, 8192, 100)
    assert np.array_equal(a["history_sample"][-1], a["state_sample"])
    assert not np.array_equal(a["history_sample"][-2], a["state_sample"])
    assert np.all(np.isfinite(a["state_sample"])) and np.all(np.isfinite(a["lnl"]))
    # 4 timed generations of 10^5 chains: every chain-step is counted once (plus the reference's initial 1 rejected)
    assert a["accepted_rejected"].sum() == 4 * 100000 + 1
    for k in a:
        assert np.array_equal(a[k], b[k]), k
