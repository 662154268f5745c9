"""CPU: the bench.py contract line of the reference arm (`--impl reference`: the oracle port on the host cores) on a
tiny configuration — the keys the driver reads must be present and well-formed without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, BENCH_N="250000", BENCH_Q="2", BENCH_R="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("queries/sec (embed+top-k+rerank)")
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["scaling"] == "strong"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_caps_the_size_with_a_fixed_row_sample(tmp_path, monkeypatch):
    import numpy as np

    import bench
    ids = np.arange(4000, dtype=np.float64).reshape(400, 10)
    sc = -ids.astype(np.float32)
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 10 * (8 + 4))
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), {"ids": ids, "scores": sc})
    a_ids, a_sc = np.load(tmp_path / "a" / "ids.npy"), np.load(tmp_path / "a" / "scores.npy")
    assert a_ids.shape == a_sc.shape == (100, 10) and a_ids.nbytes + a_sc.nbytes <= bench.DUMP_BYTES
    rows = (a_ids[:, 0] // 10).astype(int)
    assert (np.diff(rows) > 0).all() and (a_ids == ids[rows]).all() and (a_sc == sc[rows]).all()
    assert np.array_equal(a_ids, np.load(tmp_path / "b" / "ids.npy"))
    bench.dump_outputs(str(tmp_path / "small"), {"ids": ids[:5], "scores": sc[:5]})      # under the cap: every row
    assert np.array_equal(np.load(tmp_path / "small" / "ids.npy"), ids[:5])
