"""bench.py's reference arm (the CPU port of the path, no GPU needed) prints exactly one JSON line with the contract keys."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--files", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "scanned rows/s" and d["unit"] == "rows/s" and d["higher_is_better"] is True
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["config"]["workload"].startswith("config2") and d["config"]["codec"] == "snappy"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and "sample" in cb       # one SST -> one busy thread
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--files", "1", "--steps", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dumped_outputs_are_the_packed_groups(tmp_path, monkeypatch):
    import bench
    f = lambda a: np.array(a, dtype=np.float64).view(np.int64)
    block = np.array([[7, 9, 0], [0, 0, 0], [2, 1, 0], f([1.5, -0.0, 0]), f([0.5, -0.0, 0]), f([1.0, -0.0, 0])], dtype=np.int64)
    cols = bench.unpack_outputs(block)                 # the third column pads (count 0)
    assert sorted(cols) == ["count", "max", "min", "series_id", "sum"]
    assert cols["series_id"].tolist() == [7, 9] and cols["count"].tolist() == [2, 1] and cols["sum"].tolist() == [1.5, 0.0]
    assert np.signbit(cols["sum"][1]) and cols["min"].tolist() == [0.5, -0.0] and cols["max"].tolist() == [1.0, -0.0]
    bench.dump_outputs(str(tmp_path / "all"), cols)
    assert sorted(os.listdir(tmp_path / "all")) == ["count.npy", "max.npy", "min.npy", "series_id.npy", "sum.npy"]
    assert np.load(tmp_path / "all" / "sum.npy").dtype == np.float64
    # above the size limit: the same seeded sample every time, with the rows it holds
    n = 1000
    big = {k: np.arange(n, dtype=np.float64) * (i + 1) for i, k in enumerate(("series_id", "count", "sum", "min", "max"))}
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 6 * 8 * 116)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big)
    idx = np.load(tmp_path / "a" / "row_index.npy")
    assert len(idx) == 100 and np.all(np.diff(idx) > 0)
    for k in ("row_index", *big):
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "sum.npy"), idx * 3)
    assert sum(os.path.getsize(tmp_path / "a" / x) for x in os.listdir(tmp_path / "a")) <= 6 * 8 * 116


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_result(tmp_path):
    """`--dump-outputs` on one SST: the arrays written are the oracle's per-series answer for that file, bit for bit."""
    out = tmp_path / "out"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--files", "1", "--steps", "2", "--warmup", "1", "--e2e-steps", "1",
                        "--no-variant", "--no-compaction", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["parity"]["ok"] is True
    import bench
    from horaedb_b200 import sstgen
    from oracle import oracle
    _, data, _ = bench._gen_file((0, 1_000_000, "snappy"))     # rank 0's first file, as bench.py generates it
    exp = oracle.scan_aggregate([data], sstgen.metric_storage_schema().arrow_schema, 2, bench.preds(), group_col=0, value_col=2)
    got = {k: np.load(out / f"{k}.npy") for k in ("series_id", "count", "sum", "min", "max")}
    assert len(got["count"]) == len(exp.count) > 0
    assert np.array_equal(got["series_id"], exp.gkey.astype(np.float64)) and np.array_equal(got["count"], exp.count.astype(np.float64))
    for k in ("sum", "min", "max"):
        assert np.array_equal(got[k].view(np.int64), np.asarray(getattr(exp, k), dtype=np.float64).view(np.int64)), k
