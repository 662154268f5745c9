"""GPU: `bench.py --dump-outputs` writes the result of the last timed step, and the same arguments dump the same values
(the property that lets two builds be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, Q, R = 250_000, 4, 16


def _bench(out_dir):
    env = dict(os.environ, BENCH_N=str(N), BENCH_Q=str(Q), BENCH_R=str(R))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def test_dump_outputs_hold_the_reranked_top10_and_repeat(cuda, tmp_path):
    d = _bench(tmp_path / "a")
    assert d["steps"] == 2 and d["warmup"] == 1
    ids, sc = np.load(tmp_path / "a" / "ids.npy"), np.load(tmp_path / "a" / "scores.npy")
    assert ids.dtype == np.float64 and sc.dtype == np.float32 and ids.shape == sc.shape == (Q, 10)
    assert (ids == np.round(ids)).all() and ids.min() >= 0 and ids.max() < N
    assert all(len(set(r.tolist())) == 10 for r in ids)
    assert np.isfinite(sc).all() and (np.diff(sc, axis=1) <= 0).all()          # best logit first
    _bench(tmp_path / "b")
    for name in ("ids", "scores"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")), name
