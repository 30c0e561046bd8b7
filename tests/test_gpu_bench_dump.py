"""bench.py --dump-outputs end to end: the dump is the state the timed iterations leave (the same state bench.py's state_check
summarises), it is float64 and under 64 MB, and two runs with the same arguments write identical files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(workload, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", workload, "--steps", "2",
                        "--warmup", "3", "--no-cpu", "--no-e2e", "--dump-outputs", out], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.parametrize("workload", ["c3shard8", "c4"])
def test_dump_is_the_timed_state(tmp_path, workload):
    import bench
    L, M, H, kind, _, _ = bench.WORKLOADS[workload]
    runs = [_bench(workload, str(tmp_path / d)) for d in ("a", "b")]
    sc = runs[0]["state_check"]
    assert runs[0]["steps"] == 2 and sc["iterations"] == 5
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) < 64e6
    out = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n, a in out.items():
        assert a.dtype == np.float64 and np.all(np.isfinite(a)), n
        assert np.array_equal(a, np.load(tmp_path / "b" / (n + ".npy"))), n

    rel = lambda a, b: abs(a - b) <= 1e-12 * abs(b)
    assert out["BHat"].shape == (L, H) and rel(float(np.linalg.norm(out["BHat"])), sc["norm_BHat_fro"])
    assert rel(float(np.trace(out["SigmaA"])), sc["trace_SigmaA"]) and rel(float(np.trace(out["SigmaB"])), sc["trace_SigmaB"])
    assert float(out["final_delta"]) == sc["delta"] == runs[0]["final_delta"]
    if kind == "dense":
        assert float(out["sigma2"]) == sc["noise"]
        assert out["AHat"].shape == (M, H) and rel(float(np.sqrt(np.sum(out["AHat"] ** 2))), sc["norm_AHat_fro"])
    else:
        assert float(out["sigmaHat"]) == sc["noise"] and rel(float(np.sum(out["CB"])), sc["sum_CB"])
        k = out["AHat"].shape[0]
        assert 0 < k < M and out["AHat"].shape == (k, H)
        assert np.array_equal(out["ATVecHat"].reshape(k, H), out["AHat"])   # the same sampled columns in every column field
