"""bench.py --dump-outputs: the headline's outputs of its last timed step, identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, steps, warmup, chains):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                        "--chains", str(chains), "--configs", "none", "--no-cpu", "--no-ess", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    return {k: np.load(out / (k + ".npy")) for k in ("draws", "positions", "grad_evals")}


def test_bench_dump_outputs_depend_only_on_the_transitions_run(cuda_lib, tmp_path):
    """2 timed steps after 1 warm-up step and 1 timed step after 2 warm-up steps both leave every chain after its third
    transition: the dumps must agree bit for bit.  5000 chains: the positions are the fixed sample of 4096 chains."""
    import bench
    n = 5000
    a = _bench(tmp_path / "a", 2, 1, n)
    b = _bench(tmp_path / "b", 1, 2, n)
    assert a["draws"].shape == (1, n, bench.MONITOR) and a["positions"].shape == (bench.DUMP_STATE_CHAINS, bench.D)
    assert all(x.dtype == np.float64 for x in a.values()) and a["grad_evals"].shape == (2,)
    assert np.isfinite(a["positions"]).all() and a["grad_evals"].sum() > n
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # a draw is the monitored coordinates of the position the step ended in
    rows = np.sort(np.random.default_rng(bench.SEED).choice(n, bench.DUMP_STATE_CHAINS, replace=False))
    assert np.array_equal(a["draws"][0, rows], a["positions"][:, :bench.MONITOR])
