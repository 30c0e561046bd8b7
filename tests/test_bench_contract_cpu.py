"""CPU checks of the bench.py contract that need no GPU: the reference arm prints one JSON line with the agreed keys, and the
logging mirror round-trips."""
import json
import os
import subprocess
import sys

import numpy as np

import vbmf_b200_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, VBMF_BENCH_CPU_BUDGET_S="3")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "iterations/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "20000x200000x64" in d["metric"] and "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_samples_columns_consistently(tmp_path, monkeypatch):
    import bench
    vb = vbmf_b200_loader.load()

    class Shape:
        shape = (30, 500)
    p = vb.vbmf_sparse_init(Shape, 4, rng=np.random.default_rng(0), trYTY=1.0)
    p.CA = np.arange(p.MH, dtype=np.float64)
    monkeypatch.setattr(bench, "DUMP_BYTES", 40000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), p, 0.25, "sparse")
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "labels.npy" not in names and "final_delta.npy" in names
    out = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert all(a.dtype == np.float64 for a in out.values())
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) < 40000 + 128 * len(names)
    for n in names:
        assert np.array_equal(out[n[:-4]], np.load(tmp_path / "b" / n))
    cols = out["CA"].reshape(-1, 4)[:, 0] // 4          # CA[m*H + h] = m*H + h names its column
    assert 0 < cols.size < 500 and np.all(np.diff(cols) > 0)
    assert np.array_equal(out["AHat"], p.AHat[cols.astype(int)]) and np.array_equal(out["ATVecHat"].reshape(-1, 4), out["AHat"])
    assert np.array_equal(out["BHat"], p.BHat) and out["final_delta"] == 0.25


def test_log_roundtrip(tmp_path):
    vb = vbmf_b200_loader.load()
    Y = np.arange(12.0).reshape(3, 4)
    p = vb.vbmf_init(Y, 2, rng=np.random.default_rng(0))
    log = vb.create_log(p)
    p.sigma2 = 0.5
    p.BHat = p.BHat + 1.0
    vb.update_log_(log, p)
    d = vb.save_log(log, Y, {}, str(tmp_path), desc="t")
    lg, Yl = vb.load_log(d)
    assert np.array_equal(Yl, Y) and lg["sigma2"].tolist() == [1.0, 0.5] and lg["BHat"].shape == (3, 2, 2)
    q = vb.vbmf_init(Y, 2, rng=np.random.default_rng(1))
    vb.extract_params_(lg, q, 1)
    assert q.sigma2 == 0.5 and np.array_equal(q.BHat, p.BHat)
