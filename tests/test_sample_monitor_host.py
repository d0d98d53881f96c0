"""Host side of sample-quality monitoring in train.fit (no GPU): the refusals of fit(sample_every=..., sample_count=...)
and of `train --sample_every / --sample_count`, made before any device work; resume points written with other
monitoring settings, and ones written before monitoring existed; and the per-crystal metric gather plus summary under
gloo at world size 2."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT

sys.path.insert(0, os.path.dirname(__file__))
from test_resume_host import _dataset, _model, _no_device_work, _splits, _write_resume_point  # noqa: E402


def test_fit_refuses_bad_monitoring_settings_before_device_work(tmp_path, monkeypatch):
    from arreau_b200.train import fit
    _, ds = _dataset(tmp_path)
    model = _model(ds)
    _no_device_work(monkeypatch, model)
    run = dict(epochs=3, batch_size=8, device="cuda", log=lambda *_: None)
    with pytest.raises(ValueError, match="sample_every must be an integer >= 0"):
        fit(model, ds, sample_every=-1, **run)
    with pytest.raises(ValueError, match="sample_count must be an integer >= 1, got 0"):
        fit(model, ds, sample_every=2, sample_count=0, **run)
    with pytest.raises(ValueError, match="sample_count must be an integer >= 1"):
        fit(model, ds, sample_count=-5, **run)


def test_resume_with_other_monitoring_settings_is_refused(tmp_path, monkeypatch):
    from arreau_b200.train import check_resume, fit
    _, ds = _dataset(tmp_path)
    tr, va = _splits(ds)
    model = _model(ds)
    _no_device_work(monkeypatch, model)
    run = dict(epochs=3, batch_size=8, device="cuda", val_dataset=va, log=lambda *_: None)
    mon = tmp_path / "mon.ckpt"
    _write_resume_point(model, mon, len(tr), len(va), sample_every=2, sample_count=24,
                        sample_quality=[{"epoch": 1, "frac_valid": 0.5}])
    cases = [({}, "sample_every: checkpoint 2, this run 0"),
             ({"sample_every": 3, "sample_count": 24}, "sample_every: checkpoint 2, this run 3"),
             ({"sample_every": 2}, "sample_count: checkpoint 24, this run 1024"),
             ({"sample_every": 2, "sample_count": 32}, "sample_count: checkpoint 24, this run 32")]
    for over, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fit(model, tr, resume_from=str(mon), **{**run, **over})
    ck = check_resume(str(mon), epochs=3, batch_size=8, world_size=1, backward_precision="tf32", num_train=len(tr),
                      num_valid=len(va), sample_every=2, sample_count=24)
    assert ck["fit_state"]["sample_quality"] == [{"epoch": 1, "frac_valid": 0.5}]


def test_resume_point_written_before_monitoring_is_a_run_without_it(tmp_path, monkeypatch):
    """A last.ckpt whose fit_state has no sample_* keys resumes as a run with monitoring off (any sample_count), and
    refuses a run that monitors."""
    from arreau_b200.lightning_wrappers.diffusion import load_checkpoint_file
    from arreau_b200.train import check_resume, fit
    _, ds = _dataset(tmp_path)
    tr, va = _splits(ds)
    model = _model(ds)
    old = tmp_path / "last.ckpt"
    _write_resume_point(model, old, len(tr), len(va))
    assert not any(k.startswith("sample") for k in load_checkpoint_file(str(old))["fit_state"])
    common = dict(epochs=3, batch_size=8, world_size=1, backward_precision="tf32", num_train=len(tr), num_valid=len(va))
    for count in (1024, 7):
        assert check_resume(str(old), sample_every=0, sample_count=count, **common)["epoch"] == 1
    with pytest.raises(ValueError, match="sample_every: checkpoint 0, this run 2"):
        check_resume(str(old), sample_every=2, **common)
    _no_device_work(monkeypatch, model)
    with pytest.raises(AssertionError, match="device work before the resume checks"):   # the checks passed
        fit(model, tr, 3, 8, "cuda", val_dataset=va, resume_from=str(old), log=lambda *_: None)


def _cli(*args):
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, "-m", "arreau_b200.train", *args], cwd=ROOT, env=env, capture_output=True,
                          text=True)


def test_cli_refuses_bad_monitoring_settings_before_device_work(tmp_path):
    path, ds = _dataset(tmp_path)
    tr, va = _splits(ds)
    base = ["--data", path, "--batch_size", "8", "--val_fraction", "0.25", "--epochs", "3"]
    out = _cli(*base, "--sample_every", "-1")
    assert out.returncode == 2 and "sample_every must be an integer >= 0" in out.stderr, out.stderr[-2000:]
    out = _cli(*base, "--sample_every", "2", "--sample_count", "0")
    assert out.returncode == 2 and "sample_count must be an integer >= 1" in out.stderr, out.stderr[-2000:]
    good = tmp_path / "last.ckpt"
    _write_resume_point(_model(ds), good, len(tr), len(va), sample_every=2, sample_count=16)
    out = _cli(*base, "--resume", str(good), "--sample_every", "2")
    assert out.returncode == 2 and "sample_count: checkpoint 16, this run 1024" in out.stderr, out.stderr[-2000:]
    out = _cli(*base, "--resume", str(good))
    assert out.returncode == 2 and "sample_every: checkpoint 2, this run 0" in out.stderr, out.stderr[-2000:]


def _metrics(G, seed):
    """A CrystalMetrics of G crystals with every kind of row (valid, unknown element, degenerate, one atom)."""
    from arreau_b200.inference.crystal_metrics import DEGENERATE, EXTENDED_SEARCH, UNKNOWN_ELEMENT, VALID, CrystalMetrics
    rng = np.random.default_rng(seed)
    flags = rng.choice([VALID, VALID, VALID | EXTENDED_SEARCH, 0, UNKNOWN_ELEMENT, DEGENERATE], G).astype(np.int32)
    na = rng.integers(1, 30, G)
    min_dist = rng.uniform(0.2, 3.0, G)
    min_dist[na == 1] = np.inf
    min_dist[(flags & DEGENERATE) != 0] = np.nan
    density = rng.uniform(1.0, 8.0, G)
    density[(flags & UNKNOWN_ELEMENT) != 0] = np.nan
    return CrystalMetrics(num_atoms=na, volume=rng.uniform(10, 900, G), min_dist=min_dist, density=density,
                          num_elements=rng.integers(1, 5, G).astype(np.int32), flags=flags)


def _gather_worker(rank, world, port, out, G):
    from arreau_b200.distributed import gather_crystal_metrics, shard_range
    from arreau_b200.inference.crystal_metrics import METRIC_FIELDS, CrystalMetrics, quality_record, summarize
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        whole = _metrics(G, 1)
        lo, hi = shard_range(G, rank, world)
        local = CrystalMetrics(**{k: getattr(whole, k)[lo:hi] for k in METRIC_FIELDS})
        rows = gather_crystal_metrics(local)
        np.savez(os.path.join(out, f"r{rank}_{G}.npz"), **{k: getattr(rows, k) for k in METRIC_FIELDS})
        if rank == 0:
            torch.save(quality_record(summarize(rows, _metrics(50, 2)), 4), os.path.join(out, f"rec_{G}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("G", [37, 1])
def test_metric_rows_gather_and_summary_world2(tmp_path, G):
    """Every rank gets the whole set's rows in crystal order, with each field's dtype; rank 0's record equals the
    summary of the undistributed set.  G = 1: rank 1 owns no crystal and still joins the gather."""
    from arreau_b200.inference.crystal_metrics import METRIC_FIELDS, QUALITY_KEYS, quality_record, summarize
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_gather_worker, args=(2, port, str(tmp_path), G), nprocs=2, join=True)
    whole = _metrics(G, 1)
    for r in range(2):
        z = np.load(tmp_path / f"r{r}_{G}.npz")
        for k in METRIC_FIELDS:
            assert z[k].dtype == getattr(whole, k).dtype and z[k].tobytes() == getattr(whole, k).tobytes(), k
    rec = torch.load(tmp_path / f"rec_{G}.pt")
    assert rec == quality_record(summarize(whole, _metrics(50, 2)), 4)
    assert list(rec) == ["epoch", *QUALITY_KEYS] and rec["epoch"] == 4
