"""CPU tests of bench.py's --dump-outputs writer and of its argument checks (the timed GPU path itself is exercised on the GPU)."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _outputs(K):
    rng = np.random.default_rng(1)
    return {"loglik": np.array([-1.5e6]), "lambda0": rng.random(K), "W": rng.random((K, K)), "A": (rng.random((K, K)) < 0.1).astype(np.float64)}


def test_dump_writes_every_output_as_float64_when_it_fits(tmp_path):
    out = _outputs(20)
    bench.dump_outputs(str(tmp_path), out)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in out)
    for k, v in out.items():
        got = np.load(tmp_path / (k + ".npy"))
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, v)


def test_dump_samples_large_outputs_to_the_same_positions_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    out = _outputs(100)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), out)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 40_000
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "lambda0.npy"), out["lambda0"])  # small outputs stay whole
    w = np.load(tmp_path / "a" / "W.npy")
    assert 0 < w.size < out["W"].size
    np.testing.assert_array_equal(w, np.load(tmp_path / "b" / "W.npy"))
    assert np.all(np.isin(w, out["W"].ravel()))


def _bench_args(*extra):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(extra), capture_output=True, text=True, timeout=120)


def test_steps_must_be_at_least_one():
    r = _bench_args("--impl", "reference", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    r = _bench_args("--impl", "reference", "--dump-outputs", str(tmp_path))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not os.listdir(tmp_path)
