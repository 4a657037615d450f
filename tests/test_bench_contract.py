"""bench.py's reference arm runs on the host cores only, so its JSON line can be checked here: the keys the driver reads,
the same metric / unit / config as the GPU arm, and a bounded CPU sample."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "parent-set local scores/sec" and d["unit"] == "sets/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["vs_baseline"] is None and d["scaling"] in ("weak", "strong")
    assert "configs[3]" in d["config"]["workload"] and d["config"]["sets_per_step"] == 1699690
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_layout_and_sample(tmp_path):
    """--dump-outputs: rows in variable order, the parent masks recoverable exactly from their 32-bit halves, and a fixed
    seeded sample of rows, in order, once the output exceeds the size limit"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(3)
    caches = {v: (rng.integers(0, 1 << 63, size=(n, 2), dtype=np.uint64), rng.normal(size=n).astype(np.float32))
              for v, n in ((2, 5), (0, 7), (1, 0))}
    bench.dump_outputs(str(tmp_path / "all"), caches)
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in ("variable", "parents", "scores", "index")}
    assert got["parents"].dtype == got["variable"].dtype == got["index"].dtype == np.float64 and got["scores"].dtype == np.float32
    assert got["variable"].tolist() == [0] * 7 + [2] * 5 and got["index"].tolist() == list(range(12))
    p = got["parents"].astype(np.uint64)
    masks = p[:, 0::2] | (p[:, 1::2] << np.uint64(32))
    assert np.array_equal(masks, np.concatenate([caches[0][0], caches[2][0]]))
    assert np.array_equal(got["scores"], np.concatenate([caches[0][1], caches[2][1]]))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), caches, limit=4 * 128 + 5 * (8 + 32 + 4 + 8))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 4 * 128 + 5 * (8 + 32 + 4 + 8)
    idx = np.load(tmp_path / "a" / "index.npy")
    assert len(idx) == 5 and np.all(np.diff(idx) > 0) and np.array_equal(idx, np.load(tmp_path / "b" / "index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), np.concatenate([caches[0][1], caches[2][1]])[idx.astype(int)])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
