"""bench.py without a GPU: --dump-outputs writes float32 / float64 .npy files within its size limit, sampling the same
rows of every large array, and arguments that contradict each other are refused before anything runs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _arrays(N, G):
    rng = np.random.default_rng(0)
    return {"frac": rng.standard_normal((N, 3)), "types": rng.integers(0, 90, N), "score": rng.standard_normal((N, 3)).astype(np.float32),
            "logits": rng.standard_normal((N, 90)).astype(np.float32), "lengths": rng.standard_normal((G, 3)),
            "loss": np.arange(5.0)}


def test_dump_outputs_writes_every_array_whole_below_the_limit(tmp_path):
    import bench
    arrays = _arrays(4000, 100)
    bench.dump_outputs(str(tmp_path), arrays)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in arrays)
    for k, a in arrays.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == (a.dtype if a.dtype in (np.float32, np.float64) else np.float64), k
        assert np.array_equal(got, a), k


def test_dump_outputs_samples_the_same_rows_above_the_limit(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT", 2_000_000)
    arrays = _arrays(8000, 100)
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_LIMIT
    frac, types = np.load(tmp_path / "a" / "frac.npy"), np.load(tmp_path / "a" / "types.npy")
    rows = np.flatnonzero(np.isin(arrays["frac"][:, 0], frac[:, 0]))
    assert 0 < len(rows) < 8000 and np.array_equal(arrays["frac"][rows], frac)
    for k in ("types", "score", "logits"):                       # every per-atom array keeps the same rows
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), arrays[k][rows]), k
    for k in ("lengths", "loss"):                                # small arrays are written whole
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), arrays[k]), k
    for f in os.listdir(tmp_path / "a"):                         # same arguments, same sample
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    assert types.dtype == np.float64


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--trajectory", "--steps", "5"],
                                  ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_contradictory_arguments(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error:" in r.stderr, r.stderr
