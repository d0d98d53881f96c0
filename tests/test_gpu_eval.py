"""Forward-only loss evaluation (arreau_eval_noise, arreau_eval_loss, EvalEngine, DiffusionLoss.evaluate,
evaluation.evaluate_dataset, train.fit's validation and checkpoints, the training CLI's splits) on the GPU.

Tolerances: the fp32 path against the live reference (tests/golden/train_c5small.npz) within north_star's 1e-4; the
per-batch rebuild from the per-crystal sums against arreau_training_loss's loss_out within 1e-13 (only the summation
order differs); per-atom terms bit-identical.  fp16 tcgen05 path: loss and its four parts within TOL_FP16_EVAL of
max(|ref|, 1e-3) (measured on a B200: see the constant)."""
import argparse
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu
T, Z = 1000, 90
PARTS = ("loss", "e_frac", "vb", "ce", "e_lat")
# fp16 tensor path against the fp64 reference loss and its parts on both golden cases, relative to max(|ref|, 1e-3);
# measured on a B200 (1000 W): loss 1.6e-4, e_frac 1.2e-5, vb 1.6e-5, ce 1.6e-6, e_lat 3.1e-4
TOL_FP16_EVAL = 1e-3


def _case(z, case):
    p = f"{case}/"
    return {k[len(p):]: z[k] for k in z.files if k.startswith(p)}


def _rebuild(num_atoms, terms):
    """arreau_training_loss's loss_out of ONE batch from the per-crystal sums."""
    from arreau_b200.training import HYBRID_LOSS_COEFF
    terms = np.asarray(terms, dtype=np.float64)
    N, G = float(np.sum(num_atoms)), terms.shape[0]
    e_frac, vb, ce = terms[:, 0].sum() / N, terms[:, 1].sum() / N, terms[:, 2].sum() / N
    e_lat = terms[:, 3].sum() / (3.0 * G)
    return np.array([e_frac + (vb * HYBRID_LOSS_COEFF + ce) + e_lat, e_frac, vb, ce, e_lat])


def _mirror(device, weights_npz, precision):
    from arreau_b200.diffusion.diffusion_helpers import GaussianFourierProjection
    from arreau_b200.diffusion.diffusion_loss import DiffusionLoss
    from arreau_b200.ponita.models.ponita import PonitaFiberBundle
    net = PonitaFiberBundle(164 + 4, 128, Z, 3, 0, 0, 5, output_dim_vec=1, radius=5.0, num_ori=16, basis_dim=256,
                            degree=3, widening_factor=4, layer_scale=1e-6, multiple_readouts=True,
                            ori_grid=weights_npz["ori_grid"], precision=precision)
    net.load_state_dict({k: torch.as_tensor(weights_npz[k]) for k in weights_npz.files if k not in ("ori_grid", "fourier_w")})
    temb = GaussianFourierProjection(32, 16)
    with torch.no_grad():
        temb.gaussian_fourier_proj_w.copy_(torch.as_tensor(weights_npz["fourier_w"]))
    dl = DiffusionLoss(argparse.Namespace(radius=5.0, max_neighbors=8, num_timesteps=T), Z, precision=precision)
    return net.to(device), temb, dl


def _batch(c, device):
    return argparse.Namespace(X0=torch.as_tensor(c["frac0"]).to(device), A0=torch.as_tensor(c["types0"]).to(device),
                              L0=torch.as_tensor(c["lattice0"]).reshape(-1, 3).to(device),
                              num_atoms=torch.as_tensor(c["num_atoms"]).to(device))


def _noise(c, device):
    return tuple(torch.as_tensor(c[k]).to(device) for k in ("eps_x", "u", "eps_l"))


@pytest.mark.parametrize("case", [0, 1])
def test_fp32_evaluate_matches_reference_and_training_loss(device, gold, weights_npz, case):
    from arreau_b200.evaluation import EvalEngine
    from arreau_b200.tables import build_tables
    from arreau_b200.training import FlatParams, TrainEngine
    c = _case(gold("train_c5small.npz"), case)
    G = len(c["num_atoms"])
    # the public face against the live reference
    net, temb, dl = _mirror(device, weights_npz, "fp32")
    r = dl.evaluate(net, _batch(c, device), temb, np.arange(G), timestep=torch.as_tensor(c["timestep"]).reshape(-1),
                    noise=_noise(c, device))
    assert np.array_equal(r.t.cpu().numpy(), np.asarray(c["timestep"]).reshape(-1))
    got = _rebuild(c["num_atoms"], r.terms.cpu().numpy())
    for i, k in enumerate(PARTS):
        assert abs(got[i] - float(c[k])) <= 1e-4 * max(abs(float(c[k])), 1e-3), (k, got[i], float(c[k]))
    # the training step on the same weights and draws: identical per-atom terms, loss_out rebuilt to 1e-13
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    p = FlatParams(164, 4, Z, device)
    p.load_state_dict(sd)
    tabs = build_tables(T, Z)
    te = TrainEngine(p, tabs, weights_npz["fourier_w"], weights_npz["ori_grid"], c["num_atoms"], 5.0, 8, device=device)
    loss, _ = te.loss_and_grads(c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    ee = EvalEngine(te.w, tabs, weights_npz["fourier_w"], c["num_atoms"], 5.0, 8, device=device)
    _, per_crystal = ee.run(torch.as_tensor(c["frac0"]).to(device), torch.as_tensor(c["types0"]).to(device),
                            torch.as_tensor(c["lattice0"]).to(device), np.arange(G), timestep=c["timestep"],
                            noise=_noise(c, device))
    assert torch.equal(ee.terms, te.terms)
    want = loss.cpu().numpy()
    got = _rebuild(c["num_atoms"], per_crystal.cpu().numpy())
    assert np.all(np.abs(got - want) <= 1e-13 * np.abs(want)), (got, want)


def test_fp16_evaluate_matches_reference(device, gold, weights_npz):
    net, temb, dl = _mirror(device, weights_npz, "fp16")
    worst = {}
    for case in (0, 1):
        c = _case(gold("train_c5small.npz"), case)
        r = dl.evaluate(net, _batch(c, device), temb, np.arange(len(c["num_atoms"])),
                        timestep=torch.as_tensor(c["timestep"]).reshape(-1), noise=_noise(c, device))
        got = _rebuild(c["num_atoms"], r.terms.cpu().numpy())
        for i, k in enumerate(PARTS):
            err = abs(got[i] - float(c[k])) / max(abs(float(c[k])), 1e-3)
            worst[k] = max(worst.get(k, 0.0), err)
    print("fp16 evaluate: worst relative error per part", worst)
    assert max(worst.values()) < TOL_FP16_EVAL, worst


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


def _model(ds, precision="fp32", **over):
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import default_args
    torch.manual_seed(0)
    return PONITA_DIFFUSION(default_args(**over), ds.z_table, precision=precision)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_valid_loss_is_independent_of_gpu_batch(device, tmp_path, precision):
    from arreau_b200.diffusion.lattice_dataset import CrystalSubset, split_indices
    from arreau_b200.evaluation import evaluate_dataset
    _, ds = _dataset(tmp_path, 400, seed=11)
    val = CrystalSubset(ds, split_indices(len(ds), [0.25, 0.75], seed=1)[1])          # 300 crystals
    model = _model(ds, precision)
    res = [evaluate_dataset(model, val, 64, device, seed=5, gpu_batch=gb) for gb in (17, 128, 300)]
    for r in res[1:]:
        assert np.array_equal(r["terms"], res[0]["terms"]) and np.array_equal(r["t"], res[0]["t"])
        assert all(r[k] == res[0][k] for k in PARTS)
    assert np.isfinite(res[0]["loss"]) and res[0]["terms"].shape == (300, 4)
    other = evaluate_dataset(model, val, 64, device, seed=6)
    assert not np.array_equal(other["t"], res[0]["t"])


def _draw(device, seed, na, ids):
    from arreau_b200 import _lib
    na = np.asarray(na)
    G, N = len(na), int(na.sum())
    off = torch.as_tensor(np.concatenate([[0], np.cumsum(na)]), dtype=torch.int32, device=device)
    coa = torch.as_tensor(np.repeat(np.arange(G), na), dtype=torch.int32, device=device)
    ids = torch.as_tensor(ids, dtype=torch.int64, device=device)
    t = torch.zeros(G, dtype=torch.int32, device=device)
    eps_x, u = torch.zeros(N, 3, dtype=torch.float64, device=device), torch.zeros(N, Z, dtype=torch.float64, device=device)
    eps_l = torch.zeros(G, 3, dtype=torch.float64, device=device)
    _lib.call("arreau_eval_noise", seed, G, N, Z, T, ids.data_ptr(), off.data_ptr(), coa.data_ptr(), t.data_ptr(),
              eps_x.data_ptr(), u.data_ptr(), eps_l.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return t.cpu().numpy(), eps_x.cpu().numpy(), u.cpu().numpy(), eps_l.cpu().numpy()


def test_eval_noise_is_keyed_per_crystal(device):
    rng = np.random.default_rng(0)
    na = rng.integers(1, 12, 40)
    ids = rng.permutation(10 ** 6)[:40]
    a, b, c = _draw(device, 7, na, ids), _draw(device, 7, na, ids), _draw(device, 8, na, ids)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert all(not np.array_equal(x, y) for x, y in zip(a, c))
    # a crystal's draws do not depend on its batch: crystals 5.. alone, in a different batch
    off = np.concatenate([[0], np.cumsum(na)])
    d = _draw(device, 7, na[5:9], ids[5:9])
    assert np.array_equal(d[0], a[0][5:9]) and np.array_equal(d[3], a[3][5:9])
    assert np.array_equal(d[1], a[1][off[5]:off[9]]) and np.array_equal(d[2], a[2][off[5]:off[9]])
    # distributions: t ~ U{1..T}, eps ~ N(0,1), u ~ U[0,1)
    G = 50000
    t, eps_x, u, eps_l = _draw(device, 1, np.ones(G, dtype=np.int64), np.arange(G))
    assert t.min() == 1 and t.max() == T and len(np.unique(t)) == T
    assert abs(t.mean() - (T + 1) / 2) < 5
    for e in (eps_x.ravel(), eps_l.ravel()):
        assert abs(e.mean()) < 0.02 and abs(e.var() - 1) < 0.02 and abs((e ** 4).mean() - 3) < 0.1
    assert u.min() >= 0 and u.max() < 1 and abs(u.mean() - 0.5) < 0.002 and abs(u.var() - 1 / 12) < 0.001


def test_fit_with_validation_has_no_side_effects_and_best_checkpoint_reloads(device, tmp_path):
    from arreau_b200.diffusion.lattice_dataset import CrystalSubset, split_indices
    from arreau_b200.evaluation import evaluate_dataset
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.train import fit
    _, ds = _dataset(tmp_path, 120, seed=4)
    tr, va = (CrystalSubset(ds, p) for p in split_indices(len(ds), [0.8, 0.2], seed=0))
    runs = []
    for val in (None, va):
        model = _model(ds, lr=1e-3, epochs=2)
        metrics = {}
        hist = fit(model, tr, epochs=2, batch_size=16, device=device, log=lambda *_: None, val_dataset=val,
                   checkpoint_dir=str(tmp_path / ("ck_val" if val is not None else "ck")), metrics=metrics)
        runs.append((hist, model.model.flat.data.clone(), metrics, model))
    assert runs[0][0] == runs[1][0] and torch.equal(runs[0][1], runs[1][1])
    assert runs[0][2] == {} and len(runs[1][2]["valid"]) == 2
    assert os.path.exists(tmp_path / "ck" / "last.ckpt") and not os.path.exists(tmp_path / "ck" / "best.ckpt")
    best = min(v["loss"] for v in runs[1][2]["valid"])
    m = PONITA_DIFFUSION.load_from_checkpoint(str(tmp_path / "ck_val" / "best.ckpt"))
    assert evaluate_dataset(m, va, 16, device)["loss"] == best
    last = PONITA_DIFFUSION.load_from_checkpoint(str(tmp_path / "ck_val" / "last.ckpt"))
    assert evaluate_dataset(last, va, 16, device)["loss"] == runs[1][2]["valid"][-1]["loss"]


def test_training_cli_with_splits_and_generate(device, tmp_path):
    path, _ = _dataset(tmp_path, 100, seed=9)
    ck = tmp_path / "c"
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-m", "arreau_b200.train", "--data", path, "--epochs", "2", "--batch_size", "16",
                          "--val_fraction", "0.2", "--test_fraction", "0.1", "--checkpoint_dir", str(ck),
                          "--out", str(tmp_path / "model.ckpt")], cwd=ROOT, env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-3000:]
    assert (ck / "last.ckpt").exists() and (ck / "best.ckpt").exists()
    assert out.stdout.count("valid loss") == 2 and "test loss" in out.stdout, out.stdout
    gen = subprocess.run([sys.executable, "-m", "arreau_b200.generate", "--model_path", str(ck / "best.ckpt"),
                          "--num_crystals", "4", "--num_atoms", "4", "--out", str(tmp_path / "gen.h5")], cwd=ROOT, env=env,
                         capture_output=True, text=True)
    assert gen.returncode == 0, gen.stderr[-3000:]
