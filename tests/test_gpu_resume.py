"""Resumable training and the EMA of the weights on the GPU: train.fit(resume_from=...) continues a run bit for bit,
the training CLI's --resume across processes, the EMA update inside arreau_adam_step against torch.optim.Adam plus the
NeMo EMA formula, and a checkpoint's optimizer state loaded into torch.optim.Adam.

Tolerances: resume, EMA on / off and the CLI round trip are bit-identical (torch.equal); the EMA against the torch
statement within TOL_EMA of max|ema|; a step of the restored FusedAdam against the restored torch.optim.Adam within the
2e-6 of test_fused_adam_matches_torch over the whole flat buffer, TOL_ADAM_YOUNG per tensor."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err

pytestmark = pytest.mark.gpu
Z = 90
# FusedAdam's EMA after three steps (the first clipped) against torch.optim.Adam + _foreach_mul_ / _foreach_add_, relative
# to max|ema|; measured on a B200 (1000 W): 1.8e-7 (2.9e-7 of its own max in the worst tensor)
TOL_EMA = 1e-6
# the same step per tensor: arreau_adam_step forms 1 - beta2 in fp32 (9.99987e-4 for 0.999), so its step deviates from
# torch's by ~6e-6 of the step itself; against a tensor only a few steps old (LayerNorm biases start at zero, so their
# magnitude is a few steps) that is ~2e-6 of max|p| (measured on a B200: 2.01e-6, interaction_layers.3.norm.bias)
TOL_ADAM_YOUNG = 1e-5


def _dataset(tmp_path, n, seed, name="d"):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    from arreau_b200.synthetic import make_crystals
    cr = make_crystals(n, 1, 20, seed=seed)
    off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
    zs = [cr.types[off[i]:off[i + 1]] % 30 + 1 for i in range(n)]
    frac = [cr.frac[off[i]:off[i + 1]] for i in range(n)]
    lat = np.stack([np.diag(cr.lengths[i]) for i in range(n)])
    path = save_dataset_npz(str(tmp_path / name), zs, lat, frac)
    return path, CrystalDataset([path])


def _model(ds, **over):
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import default_args
    torch.manual_seed(0)
    return PONITA_DIFFUSION(default_args(**over), ds.z_table)


def _cli_splits(ds, val_fraction):
    """train.main's splits (no test share)."""
    from arreau_b200.diffusion.lattice_dataset import CrystalSubset, split_indices
    parts = split_indices(len(ds), [1.0 - val_fraction, val_fraction, 0.0], seed=0)
    return CrystalSubset(ds, parts[0]), CrystalSubset(ds, parts[1])


def _weights(path):
    from arreau_b200.lightning_wrappers.diffusion import load_checkpoint_file
    return load_checkpoint_file(str(path))["state_dict"]


def _same_tensors(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def _quiet(*_):
    pass


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("ema", [None, 0.9])
@pytest.mark.parametrize("with_val", [False, True])
def test_resume_is_bit_identical(device, tmp_path, with_val, ema, precision):
    """fit for 3 epochs == fit for 2, then a new model from last.ckpt resumed to 3: weights, both Adam moments, the
    EMA, the history, the valid losses and the best*.ckpt files.  The resumed run's train engine is built from other
    batches, so it has another capacity."""
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import ema_path, fit
    _, ds = _dataset(tmp_path, 72, seed=4)
    tr, va = _cli_splits(ds, 0.25)
    val = va if with_val else None
    run = dict(batch_size=12, device=device, backward_precision=precision, val_dataset=val, ema_decay=ema, log=_quiet)
    straight, met_s = _model(ds, lr=1e-3, epochs=3), {}
    hist_s = fit(straight, tr, 3, checkpoint_dir=str(tmp_path / "a"), metrics=met_s, **run)
    first, met_1 = _model(ds, lr=1e-3, epochs=3), {}
    hist_1 = fit(first, tr, 2, checkpoint_dir=str(tmp_path / "b"), metrics=met_1, **run)
    last = str(tmp_path / "b" / "last.ckpt")
    resumed, met_r = PONITA_DIFFUSION.load_from_checkpoint(last), {}
    hist_r = fit(resumed, tr, 3, checkpoint_dir=str(tmp_path / "b"), metrics=met_r, resume_from=last, **run)

    assert hist_1 == hist_s[:2] and hist_r == hist_s and len(hist_s) == 3
    so, ro = straight._optimizer, resumed._optimizer
    assert torch.equal(resumed.model.flat.data, straight.model.flat.data)
    assert torch.equal(ro.exp_avg, so.exp_avg) and torch.equal(ro.exp_avg_sq, so.exp_avg_sq)
    assert ro.step_count == so.step_count
    if ema is not None:
        assert torch.equal(ro.ema.data, so.ema.data) and not torch.equal(ro.ema.data, resumed.model.flat.data)
    te_s = straight.diffusion_loss._train_engines
    te_r = resumed.diffusion_loss._train_engines
    caps = lambda d: [(t.eng.N_cap, t.eng.G_cap) for t in d.values()]  # noqa: E731
    print("train engine capacity (atoms, crystals): straight", caps(te_s), "resumed", caps(te_r))
    assert caps(te_s) != caps(te_r)
    names = ["last.ckpt"] + (["best.ckpt"] if with_val else [])
    for n in names + ([ema_path(n) for n in names] if ema is not None else []):
        _same_tensors(_weights(tmp_path / "a" / n), _weights(tmp_path / "b" / n))
    assert not os.path.exists(tmp_path / "b" / "best.ckpt") or with_val
    if with_val:
        assert [v["loss"] for v in met_1["valid"] + met_r["valid"]] == [v["loss"] for v in met_s["valid"]]
        assert len(met_r["valid"]) == 1
    else:
        assert met_r == {}


def test_fit_with_ema_trains_identically_and_validates_the_ema(device, tmp_path):
    from arreau_b200.evaluation import evaluate_dataset
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION, load_checkpoint_file
    from arreau_b200.train import ema_model, fit
    _, ds = _dataset(tmp_path, 100, seed=6)
    tr, va = _cli_splits(ds, 0.2)
    runs = {}
    for ema in (None, 0.9):
        model, met = _model(ds, lr=1e-3, epochs=3), {}
        ck = tmp_path / f"ck{ema}"
        hist = fit(model, tr, 3, 16, device, val_dataset=va, checkpoint_dir=str(ck), metrics=met, ema_decay=ema, log=_quiet)
        runs[ema] = (hist, model, met, ck)
    (h0, m0, met0, _), (h1, m1, met1, ck1) = runs[None], runs[0.9]
    assert h0 == h1 and torch.equal(m0.model.flat.data, m1.model.flat.data)
    assert torch.equal(m0._optimizer.exp_avg, m1._optimizer.exp_avg)
    assert torch.equal(m0._optimizer.exp_avg_sq, m1._optimizer.exp_avg_sq)
    ema_losses = [v["loss"] for v in met1["valid"]]
    assert ema_losses != [v["loss"] for v in met0["valid"]]           # the EMA weights are the ones validated
    best = min(ema_losses)
    reloaded = PONITA_DIFFUSION.load_from_checkpoint(str(ck1 / "best-EMA.ckpt"))
    assert evaluate_dataset(reloaded, va, 16, device)["loss"] == best
    ema_sd = load_checkpoint_file(str(ck1 / "last-EMA.ckpt"))["state_dict"]
    for k, v in m1._optimizer.ema.views().items():
        assert torch.equal(ema_sd["model." + k], v.cpu()), k
    assert torch.equal(load_checkpoint_file(str(ck1 / "last.ckpt"))["ema"]["state_dict"]["model.x_embedder.weight"],
                       ema_sd["model.x_embedder.weight"])
    assert all(bool(ema_sd[f"model.interaction_layers.{l}.conv.callibrated"]) for l in range(5))
    before = m1._optimizer.ema.data.clone()            # another view of the EMA leaves it as it is
    twin = ema_model(m1, device)
    assert torch.equal(twin.model.flat.data, before) and twin.model.flat is m1._optimizer.ema


def test_ema_rule_matches_torch_adam_and_nemo(device, weights_npz):
    """Three steps (the first clipped): the EMA starts at the weights before the first step and follows every step
    with ema = d * ema + (1 - d) * p (NeMo's _foreach_mul_ / _foreach_add_ on torch.optim.Adam's weights); without
    an EMA buffer (NULL) the weights and moments are bit for bit those of the step with one."""
    from arreau_b200.training import FlatParams, FusedAdam
    decay = 0.9
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    p, q = FlatParams(164, 4, Z, device), FlatParams(164, 4, Z, device)
    p.load_state_dict(sd)
    q.load_state_dict(sd)
    ref = {k: v.clone().requires_grad_(True) for k, v in p.views().items()}
    decayed = [k for k in ref if k.endswith(".weight") and ".norm." not in k]
    topt = torch.optim.Adam([{"params": [ref[k] for k in decayed], "weight_decay": 0.01},
                             {"params": [v for k, v in ref.items() if k not in decayed], "weight_decay": 0.0}], lr=3e-4)
    ema_ref = [v.detach().clone() for v in ref.values()]
    opt = FusedAdam(p, lr=3e-4, weight_decay=0.01, max_grad_norm=0.5, ema_decay=decay)
    plain = FusedAdam(q, lr=3e-4, weight_decay=0.01, max_grad_norm=0.5)
    g = torch.Generator(device="cpu").manual_seed(1)
    for step in range(3):
        grad = (torch.randn(p.total, generator=g) * (10.0 if step == 0 else 1e-4)).to(device)
        p.grad.copy_(grad)
        q.grad.copy_(grad)
        for k, v in p._views(grad).items():
            ref[k].grad = v.clone()
        torch.nn.utils.clip_grad_norm_(list(ref.values()), 0.5)
        topt.step()
        with torch.no_grad():
            torch._foreach_mul_(ema_ref, decay)
            torch._foreach_add_(ema_ref, [v.detach() for v in ref.values()], alpha=1 - decay)
        opt.step()
        plain.step()
    assert torch.equal(p.data, q.data) and torch.equal(opt.exp_avg, plain.exp_avg)
    assert torch.equal(opt.exp_avg_sq, plain.exp_avg_sq)
    got = opt.ema.views()
    worst = max(rel_err(got[k].cpu().numpy(), e.cpu().numpy()) for k, e in zip(ref, ema_ref))
    whole = max(float((got[k] - e).abs().max()) for k, e in zip(ref, ema_ref)) / float(opt.ema.data.abs().max())
    print(f"EMA vs torch.optim.Adam + NeMo: {whole:.3e} of max|ema| (worst tensor, relative to its own max: {worst:.3e})")
    assert whole < TOL_EMA
    assert not torch.equal(opt.ema.data, p.data)


def test_checkpoint_optimizer_state_loads_into_torch_adam(device, tmp_path):
    """ckpt["optimizer_states"][0] of a fit's last.ckpt in a torch.optim.Adam built from its named groups, and in a
    FusedAdam restored from the same file: one more step on the same gradients agrees within 2e-6."""
    from arreau_b200.lightning_wrappers.diffusion import load_checkpoint_file
    from arreau_b200.train import fit
    from arreau_b200.training import FusedAdam
    _, ds = _dataset(tmp_path, 40, seed=2)
    fit(_model(ds, lr=1e-3, epochs=2, weight_decay=0.01), ds, 1, 16, device, checkpoint_dir=str(tmp_path / "ck"),
        log=_quiet)
    ck = load_checkpoint_file(str(tmp_path / "ck" / "last.ckpt"))
    osd = ck["optimizer_states"][0]
    w = {k[len("model."):]: v for k, v in ck["state_dict"].items() if k.startswith("model.")}
    params = {}
    groups = []
    for gr in osd["param_groups"]:
        for k in gr["param_names"]:
            params[k] = torch.nn.Parameter(w[k].clone().to(device))
        groups.append({"params": [params[k] for k in gr["param_names"]], "param_names": gr["param_names"],
                       "weight_decay": gr["weight_decay"]})
    topt = torch.optim.Adam(groups, lr=osd["param_groups"][0]["lr"])
    topt.load_state_dict(osd)
    assert osd["param_groups"][0]["weight_decay"] == 0.01
    flat = _model(ds).model.flatten_parameters(device)
    flat.load_state_dict(w)
    opt = FusedAdam(flat, lr=osd["param_groups"][0]["lr"], weight_decay=0.01, max_grad_norm=0.5)
    opt.load_state_dict(osd)
    assert opt.step_count == ck["global_step"] > 0
    grad = (torch.randn(flat.total, generator=torch.Generator().manual_seed(3)) * 1e-4).to(device)     # not clipped
    flat.grad.copy_(grad)
    for k, v in flat._views(grad).items():
        params[k].grad = v.clone()
    torch.nn.utils.clip_grad_norm_(list(params.values()), 0.5)
    topt.step()
    opt.step()
    got = flat.data.cpu().numpy()
    want = torch.empty_like(flat.data)
    for k, v in flat._views(want).items():
        v.copy_(params[k].detach())
    want = want.cpu().numpy()
    assert rel_err(got, want) < 2e-6
    worst = max((rel_err(v.cpu().numpy(), params[k].detach().cpu().numpy()), k) for k, v in flat.views().items())
    print(f"restored FusedAdam vs restored torch.optim.Adam: {rel_err(got, want):.3e} of max|p|, worst tensor {worst}")
    assert worst[0] < TOL_ADAM_YOUNG, worst


def test_cli_resume_across_processes_matches_a_straight_run(device, tmp_path):
    """CLI run A for 3 epochs; run B: 2 epochs of fit built in-process as the CLI builds it, then `--resume last.ckpt`
    in a new process.  The --out checkpoints and their -EMA twins are equal tensor for tensor."""
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import default_args, fit
    path, ds = _dataset(tmp_path, 90, seed=9)
    env = dict(os.environ, PYTHONPATH=ROOT)
    common = ["--data", path, "--batch_size", "16", "--val_fraction", "0.2", "--ema_decay", "0.999", "--epochs", "3"]

    def cli(*args):
        out = subprocess.run([sys.executable, "-m", "arreau_b200.train", *common, *args], cwd=ROOT, env=env,
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr[-3000:]
        return out.stdout

    out_a = cli("--checkpoint_dir", str(tmp_path / "a"), "--out", str(tmp_path / "a" / "model.ckpt"))
    assert out_a.count("valid loss") == 3
    tr, va = _cli_splits(ds, 0.2)
    torch.manual_seed(0)
    model = PONITA_DIFFUSION(default_args(lr=3e-4, epochs=3, warmup=0, batch_size=16), ds.z_table)
    fit(model, tr, 2, 16, device, val_dataset=va, checkpoint_dir=str(tmp_path / "b"), ema_decay=0.999, log=_quiet)
    out_b = cli("--checkpoint_dir", str(tmp_path / "b"), "--out", str(tmp_path / "b" / "model.ckpt"),
                "--resume", str(tmp_path / "b" / "last.ckpt"))
    assert out_b.count("valid loss") == 1 and "epoch 2:" in out_b
    for n in ("model.ckpt", "model-EMA.ckpt", "best-EMA.ckpt"):
        _same_tensors(_weights(tmp_path / "a" / n), _weights(tmp_path / "b" / n))
    a, b = _weights(tmp_path / "a" / "model.ckpt"), _weights(tmp_path / "a" / "model-EMA.ckpt")
    assert not torch.equal(a["model.x_embedder.weight"], b["model.x_embedder.weight"])
    _same_tensors(b, _weights(tmp_path / "a" / "last-EMA.ckpt"))
    _same_tensors(a, _weights(tmp_path / "a" / "last.ckpt"))
