"""bench.py's command line.  The reference arm runs without a GPU (it times the reference's own CPU
scan) and its one JSON line must carry the same keys as the GPU arm's, so the two arms can be compared;
--dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-queries-per-proc", "2", "--n-codes", "60000"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout must carry exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "queries/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["warmup"] >= 3 and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_dump_outputs_caps_at_64_mb(tmp_path):
    """--dump-outputs keeps a fixed, seeded sample of the queries when the top-k would pass 64 MB."""
    import numpy as np
    import bench
    Q, k = 400_000, 10
    pos = np.arange(Q * k, dtype=np.uint32).reshape(Q, k)
    dist = pos.astype(np.float32) / 7
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), pos, pos[:, ::-1], dist)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["distances.npy", "ids.npy", "positions.npy", "query_rows.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64_000_000
    rows = np.load(tmp_path / "a" / "query_rows.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "positions.npy"), pos[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy"), pos[rows, ::-1])
    assert np.array_equal(np.load(tmp_path / "a" / "distances.npy"), dist[rows])
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)), n


@pytest.mark.gpu
def test_gpu_arm_dumps_identical_outputs_run_to_run(tmp_path):
    """Two runs with the same arguments time --steps steps each and dump the same top-k, which the
    run's own parity check has compared with the CPU scan."""
    import numpy as np
    lines = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--n-codes", "60000",
                            "--queries", "3000", "--c5-codes", "0", "--no-multi-cpp", "--cpu-baseline-queries", "50",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout))
    for d in lines:
        assert d["steps"] == 2 and d["parity"]["ok"] and d["parity"]["queries"] == 50
    for name, dtype in (("positions", np.float64), ("ids", np.float64), ("distances", np.float32)):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == dtype and a.shape == (3000, 10) and np.array_equal(a, b), name
    dist = np.load(tmp_path / "a" / "distances.npy")
    assert np.all(np.diff(dist, axis=1) >= 0)
