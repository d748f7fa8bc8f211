"""bench.py's host-side contract, checked without a GPU: the reference arm prints ONE JSON line whose `config` is the
object the B200 arm prints for the same workload (the driver compares them), and times the staged, unmodified reference
(`baseline/_ref`, tools/stage_reference.sh) when it is there."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_config_is_shared_between_the_arms():
    sys.path.insert(0, ROOT)
    import bench
    for wl, (desc, kind, G, sims) in bench.WORKLOADS.items():
        c = bench.workload_config(wl, G, sims, sims)
        assert c["workload"].startswith(wl + ":") and c["net"] == kind and c["games_per_gpu"] == G and c["sims_per_move"] == sims
        assert "l2" in c and "model" not in c
        assert c == bench.workload_config(wl, G, sims, sims)
    assert set(bench.REF_PLIES_PER_STEP) == set(bench.WORKLOADS)


def test_dump_outputs_stays_under_the_limit_with_a_repeatable_sample(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"pis": np.arange(650 * 65, dtype=np.float32).reshape(650, 65), "values": np.arange(650, dtype=np.float64)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["pis.npy", "values.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "pis.npy"), arrays["pis"])
    limit = 40000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["pis.npy", "pis_rows.npy", "values.npy", "values_rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    for f in files:
        x = np.load(tmp_path / "a" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(tmp_path / "b" / f))
    rows = np.load(tmp_path / "a" / "pis_rows.npy").astype(np.int64)
    assert len(rows) > 0 and np.array_equal(rows, np.load(tmp_path / "a" / "values_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "pis.npy"), arrays["pis"][rows])
    assert np.array_equal(np.load(tmp_path / "a" / "values.npy"), arrays["values"][rows])


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "self_play_worker.py")),
                    reason="reference not staged (tools/stage_reference.sh)")
def test_reference_arm_runs_the_staged_reference():
    sums = open(os.path.join(ROOT, "baseline", "_ref", "SHA256SUMS")).read().split()
    assert "self_play_worker.py" in sums and "MCTS_model.py" in sums
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1  # exactly one JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["value"] > 0 and d["unit"] == "sims/s" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    sys.path.insert(0, ROOT)
    import bench
    desc, kind, G, sims = bench.WORKLOADS["c2"]
    assert d["config"] == bench.workload_config("c2", G, sims, sims)
    assert "one_self_play" in d["cpu_baseline"]["sample"] and "num_threads=4" in d["cpu_baseline"]["sample"]
