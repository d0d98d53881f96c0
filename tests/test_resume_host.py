"""Host side of resumable training (no GPU): the refusals of train.fit(resume_from=...) and of `train --resume`, made
before any device work; the atomic checkpoint write; FusedAdam's state in torch.optim.Adam's layout; and the per-rank
generator state gather / restore under gloo at world size 2."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import GOLD, ROOT

REFERENCE_CKPT = os.path.join(GOLD, "reference_model.ckpt")


def _dataset(tmp_path, n=40):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    rng = np.random.default_rng(3)
    na = rng.integers(1, 7, n)
    path = save_dataset_npz(str(tmp_path / "d"), [rng.integers(1, 9, k) for k in na], np.tile(np.eye(3) * 4, (n, 1, 1)),
                            [rng.random((k, 3)) for k in na])
    return path, CrystalDataset([path])


def _splits(ds, val_fraction=0.25):
    """The CLI's split (train.main) of `ds` with a validation share and no test share."""
    from arreau_b200.diffusion.lattice_dataset import CrystalSubset, split_indices
    parts = split_indices(len(ds), [1.0 - val_fraction, val_fraction, 0.0], seed=0)
    return CrystalSubset(ds, parts[0]), CrystalSubset(ds, parts[1])


def _model(ds, epochs=3):
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import default_args
    torch.manual_seed(0)
    return PONITA_DIFFUSION(default_args(epochs=epochs, batch_size=8), ds.z_table)


def _write_resume_point(model, path, num_train, num_valid, ema_decay=None, **over):
    """A last.ckpt as train.fit writes it after epoch 1 (the optimizer and generator states are placeholders)."""
    fs = {"seed": 0, "batch_size": 8, "world_size": 1, "backward_precision": "tf32", "num_train": num_train,
          "num_valid": num_valid, "train_losses": [2.0, 1.5], "valid_losses": [2.1, 1.6], "best_valid": 1.6,
          "cuda_rng": [torch.zeros(16, dtype=torch.uint8)]}
    fs.update(over)
    state = {"epoch": 1, "global_step": 8, "optimizer_states": [{"state": {}, "param_groups": []}],
             "ema": None if ema_decay is None else {"decay": ema_decay, "state_dict": {}}, "fit_state": fs}
    model.save_checkpoint(str(path), training_state=state)


def _no_device_work(monkeypatch, model):
    def boom(*a, **k):
        raise AssertionError("device work before the resume checks")
    monkeypatch.setattr(model, "to", boom)
    monkeypatch.setattr(model, "configure_optimizers", boom)


def test_fit_refuses_a_resume_point_of_another_run_before_device_work(tmp_path, monkeypatch):
    from arreau_b200.train import fit
    _, ds = _dataset(tmp_path)
    tr, va = _splits(ds)
    model = _model(ds)
    _no_device_work(monkeypatch, model)
    good = tmp_path / "last.ckpt"
    _write_resume_point(model, good, len(tr), len(va))
    plain = tmp_path / "best.ckpt"
    model.save_checkpoint(str(plain))
    run = dict(epochs=3, batch_size=8, device="cuda", val_dataset=va, log=lambda *_: None)

    for path in (plain, REFERENCE_CKPT):                     # model-only checkpoints: nothing to resume
        with pytest.raises(ValueError, match="no training state"):
            fit(model, tr, resume_from=str(path), **run)
    cases = [({"batch_size": 16}, "batch_size: checkpoint 8, this run 16"),
             ({"backward_precision": "fp32"}, "backward_precision: checkpoint tf32, this run fp32"),
             ({"epochs": 4}, "epochs: checkpoint 3, this run 4"),
             ({"val_dataset": None}, f"valid split size: checkpoint {len(va)}, this run 0"),
             ({"ema_decay": 0.999}, "ema_decay: checkpoint None, this run 0.999"),
             ({"seed": 1}, "seed: checkpoint 0, this run 1")]
    for over, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fit(model, tr, resume_from=str(good), **{**run, **over})
    with pytest.raises(ValueError, match=f"train split size: checkpoint {len(tr)}, this run {len(ds)}"):
        fit(model, ds, resume_from=str(good), **run)
    # a run at another world size, and with another EMA decay
    _write_resume_point(model, tmp_path / "w2.ckpt", len(tr), len(va), world_size=2)
    with pytest.raises(ValueError, match="world size: checkpoint 2, this run 1"):
        fit(model, tr, resume_from=str(tmp_path / "w2.ckpt"), **run)
    _write_resume_point(model, tmp_path / "ema.ckpt", len(tr), len(va), ema_decay=0.99)
    with pytest.raises(ValueError, match="ema_decay: checkpoint 0.99, this run 0.999"):
        fit(model, tr, resume_from=str(tmp_path / "ema.ckpt"), ema_decay=0.999, **run)
    with pytest.raises(ValueError, match="ema_decay: checkpoint 0.99, this run None"):
        fit(model, tr, resume_from=str(tmp_path / "ema.ckpt"), **run)


def _cli(*args):
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, "-m", "arreau_b200.train", *args], cwd=ROOT, env=env, capture_output=True,
                          text=True)


def test_cli_refuses_resume_before_device_work(tmp_path):
    """CUDA is hidden from the CLI: a refusal must come from the checks, not from the missing device."""
    path, ds = _dataset(tmp_path)
    tr, va = _splits(ds)
    model = _model(ds)
    good = tmp_path / "last.ckpt"
    _write_resume_point(model, good, len(tr), len(va))
    base = ["--data", path, "--batch_size", "8", "--val_fraction", "0.25", "--epochs", "3"]
    out = _cli(*base, "--resume", REFERENCE_CKPT)
    assert out.returncode == 2 and "no training state" in out.stderr, out.stderr[-2000:]
    out = _cli(*base[:-1], "4", "--resume", str(good))
    assert out.returncode == 2 and "epochs: checkpoint 3, this run 4" in out.stderr, out.stderr[-2000:]
    out = _cli(*base[:4], "--val_fraction", "0.5", "--epochs", "3", "--resume", str(good))
    assert out.returncode == 2 and "valid split size" in out.stderr, out.stderr[-2000:]
    out = _cli(*base, "--resume", str(good), "--lr", "1e-3")
    assert out.returncode == 2 and "--lr 0.001 differs from the resumed run's 0.0003" in out.stderr, out.stderr[-2000:]
    out = _cli(*base, "--ema_decay", "1.5")
    assert out.returncode == 2 and "--ema_decay must be in [0, 1]" in out.stderr, out.stderr[-2000:]


def test_checkpoint_write_is_atomic(tmp_path, monkeypatch):
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION, load_checkpoint_file
    _, ds = _dataset(tmp_path)
    model = _model(ds)
    path = tmp_path / "last.ckpt"
    model.save_checkpoint(str(path))
    before = path.read_bytes()
    real_save = torch.save

    def dies_mid_write(obj, f, *a, **k):
        real_save(obj, f, *a, **k)
        f.truncate(f.tell() // 2)                 # half a file on disk, then the process "dies"
        raise KeyboardInterrupt

    with torch.no_grad():
        next(model.parameters()).add_(1.0)
    monkeypatch.setattr(torch, "save", dies_mid_write)
    with pytest.raises(KeyboardInterrupt):
        model.save_checkpoint(str(path), training_state={"epoch": 5})
    monkeypatch.undo()
    assert path.read_bytes() == before
    assert [p for p in os.listdir(tmp_path) if p.endswith(".tmp")] == []
    assert "epoch" not in load_checkpoint_file(str(path))
    PONITA_DIFFUSION.load_from_checkpoint(str(path))
    # and a completed write replaces it, with the training state as extra keys
    model.save_checkpoint(str(path), training_state={"epoch": 5})
    ck = load_checkpoint_file(str(path))
    assert ck["epoch"] == 5 and {"state_dict", "hyper_parameters", "ori_grid"} <= set(ck)


def _flat_adam(ema_decay=None, weight_decay=0.01):
    from arreau_b200.training import FlatParams, FusedAdam
    p = FlatParams(40, 4, 30, "cpu")
    g = torch.Generator().manual_seed(0)
    p.data.copy_(torch.randn(p.total, generator=g))
    opt = FusedAdam(p, lr=3e-4, weight_decay=weight_decay, ema_decay=ema_decay)
    opt.exp_avg.copy_(torch.randn(p.total, generator=g))
    opt.exp_avg_sq.copy_(torch.rand(p.total, generator=g))
    opt.step_count = 7
    return p, opt


def test_fused_adam_state_dict_is_torch_adams_layout():
    p, opt = _flat_adam(ema_decay=0.999)
    opt.ema_initialized = True
    sd = opt.state_dict()
    g0, g1 = sd["param_groups"]
    assert g0["weight_decay"] == 0.01 and g1["weight_decay"] == 0.0
    decayed = [k for k in p.specs if k.endswith(".weight") and ".norm." not in k]       # FlatParams.decay_mask
    assert g0["param_names"] == decayed and g1["param_names"] == [k for k in p.specs if k not in decayed]
    assert g0["params"] + g1["params"] == list(range(len(p.specs)))
    assert sd["ema"] == {"decay": 0.999, "initialized": True}
    views_m, views_v = p._views(opt.exp_avg), p._views(opt.exp_avg_sq)
    for g in (g0, g1):
        for i, k in zip(g["params"], g["param_names"]):
            st = sd["state"][i]
            assert float(st["step"]) == 7.0 and torch.equal(st["exp_avg"], views_m[k]) and torch.equal(st["exp_avg_sq"], views_v[k])
    # it loads into a torch.optim.Adam built from the named groups ...
    ref = {k: torch.nn.Parameter(v.clone()) for k, v in p.views().items()}
    topt = torch.optim.Adam([{"params": [ref[k] for k in g["param_names"]], "param_names": g["param_names"],
                              "weight_decay": g["weight_decay"]} for g in (g0, g1)], lr=3e-4)
    topt.load_state_dict(sd)
    k = g0["param_names"][3]
    assert torch.equal(topt.state[ref[k]]["exp_avg"], views_m[k])
    # ... and back by name, whatever the order of the groups' entries
    p2, opt2 = _flat_adam(ema_decay=0.999)
    opt2.exp_avg.zero_(), opt2.exp_avg_sq.zero_()
    opt2.step_count = 0
    shuffled = {"state": {}, "param_groups": [], "ema": sd["ema"]}
    for g in reversed(sd["param_groups"]):
        order = list(reversed(range(len(g["params"]))))
        ids = [1000 + g["params"][j] for j in order]
        shuffled["param_groups"].append({**g, "params": ids, "param_names": [g["param_names"][j] for j in order]})
        for j, i in zip(order, ids):
            shuffled["state"][i] = sd["state"][g["params"][j]]
    v0, ev0 = p2.version, opt2.ema.version
    opt2.load_state_dict(shuffled)
    assert torch.equal(opt2.exp_avg, opt.exp_avg) and torch.equal(opt2.exp_avg_sq, opt.exp_avg_sq)
    assert opt2.step_count == 7 and opt2.ema_initialized and p2.version > v0 and opt2.ema.version > ev0


def test_fused_adam_load_refuses_foreign_state():
    _, opt = _flat_adam()
    sd = opt.state_dict()
    lightning = {"state": sd["state"], "param_groups": [{k: v for k, v in g.items() if k != "param_names"}
                                                        for g in sd["param_groups"]]}
    with pytest.raises(ValueError, match="no param_names"):
        opt.load_state_dict(lightning)
    renamed = {**sd, "param_groups": [dict(sd["param_groups"][0], param_names=["x"] + sd["param_groups"][0]["param_names"][1:]),
                                      sd["param_groups"][1]]}
    with pytest.raises(ValueError, match="does not name this model's parameters"):
        opt.load_state_dict(renamed)
    _, with_ema = _flat_adam(ema_decay=0.9)
    with pytest.raises(ValueError, match="EMA decay None, this optimizer 0.9"):
        with_ema.load_state_dict(sd)
    with pytest.raises(ValueError, match="ema_decay must be in"):
        _flat_adam(ema_decay=1.5)


def _rng_worker(rank, world, port, out):
    from arreau_b200.distributed import gather_rng_states, rank_rng_state
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(100 + rank)
        torch.randn(3 + rank)
        own = torch.get_rng_state()
        states = gather_rng_states(own)             # every rank joins; rank 0 is the one that writes
        if rank == 0:
            torch.save(states, os.path.join(out, "states.pt"))
        want = torch.randn(5)                        # what this rank draws next
        torch.randn(11)
        dist.barrier()
        torch.set_rng_state(rank_rng_state(torch.load(os.path.join(out, "states.pt"))))
        got = torch.randn(5)
        np.savez(os.path.join(out, f"r{rank}.npz"), own=own.numpy(), want=want.numpy(), got=got.numpy())
    finally:
        dist.destroy_process_group()


def test_rng_states_gather_to_rank0_and_restore_per_rank(tmp_path):
    from arreau_b200.distributed import gather_rng_states, rank_rng_state
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rng_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    states = torch.load(tmp_path / "states.pt")
    assert len(states) == 2 and all(st.dtype == torch.uint8 for st in states)
    for r in range(2):
        z = np.load(tmp_path / f"r{r}.npz")
        assert np.array_equal(states[r].numpy(), z["own"])
        assert np.array_equal(z["got"], z["want"])
    assert not np.array_equal(states[0].numpy(), states[1].numpy())
    # world size 1: the state itself; a list of another world size is refused
    st = torch.get_rng_state()
    assert torch.equal(rank_rng_state(gather_rng_states(st)), st)
    with pytest.raises(ValueError, match="2 ranks cannot be restored at world size 1"):
        rank_rng_state(states)
