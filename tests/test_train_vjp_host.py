"""The oracle's vector-Jacobian product of the network (oracle/training.py: ponita_vjp) and the gradient block partition
that tests/test_gpu_train_vjp.py compares the GPU backward by.  CPU only.

ponita_vjp sums the gradients of whole-crystal slices; here it must equal one autograd pass over the whole batch for
every slice size, and with the loss's own output cotangents it must reproduce training_grads, which
tests/test_oracle_training.py pins to the live reference."""
import numpy as np
import pytest
import torch

from conftest import f64_default, rel_err

T, Z, F = 1000, 90, 164


def _weights(weights_npz, radius=5.0):
    from oracle import restatement as R
    sd = {k: torch.as_tensor(weights_npz[k], dtype=torch.float64) for k in weights_npz.files
          if k not in ("ori_grid", "fourier_w")}
    return (R.PonitaWeights(sd, torch.as_tensor(weights_npz["ori_grid"], dtype=torch.float64), radius),
            torch.as_tensor(weights_npz["fourier_w"], dtype=torch.float64))


def _state(seed=3):
    """A small noised state: 7 crystals of 1..8 atoms, some atoms in the mask state, per-atom timesteps."""
    from arreau_b200.synthetic import make_crystals
    cr = make_crystals(7, 1, 8, seed=seed)
    rng = np.random.default_rng(seed)
    types = cr.types.copy()
    types[rng.random(cr.total_atoms) < 0.3] = Z - 1
    t_atom = np.repeat(rng.integers(1, T + 1, cr.num_crystals), cr.num_atoms)
    return (torch.as_tensor(cr.frac), torch.as_tensor(types), torch.as_tensor(t_atom), torch.as_tensor(cr.num_atoms),
            torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles))


@pytest.mark.parametrize("slice_crystals", [1, 3, None])
def test_chunked_vjp_equals_one_autograd_pass(weights_npz, slice_crystals):
    from oracle import restatement as R, training as TR
    with f64_default():
        W, fw = _weights(weights_npz)
        tabs = R.DiffusionTables.build(T, Z)
        frac, types, t_atom, na, lengths, angles = _state()
        N, G = frac.shape[0], na.shape[0]
        g = torch.Generator().manual_seed(11)
        cots = [(torch.randn(N, 3, generator=g), torch.randn(N, Z, generator=g), torch.randn(G, 3, generator=g)),
                (torch.randn(N, 3, generator=g), None, None), (None, None, torch.randn(G, 3, generator=g))]
        outs, grads, ei = TR.ponita_vjp(W, tabs, fw, frac, types, t_atom, na, lengths, angles, 5.0, 8, cots,
                                        slice_crystals=slice_crystals)
        # the whole batch in one forward, autograd of <cot, outputs> directly
        leaves = {k: v.clone().requires_grad_(True) for k, v in W.sd.items()}
        W2 = R.PonitaWeights(leaves, W.ori_grid, W.radius)
        onehot = torch.nn.functional.one_hot(types, Z).double()
        score, logits, len0, graph = R.predict_scores(W2, tabs, fw, frac, onehot, t_atom, na, lengths, angles, 5.0, 8,
                                                      return_graph=True)
        assert torch.equal(ei[0], graph[0]) and torch.equal(ei[1], graph[1])
        for got, ref in zip((outs["score"], outs["logits"], outs["len0"]), (score, logits, len0)):
            assert rel_err(got.numpy(), ref.detach().numpy()) < 1e-12
        for i, cot in enumerate(cots):
            obj = sum((y * c).sum() for y, c in zip((score, logits, len0), cot) if c is not None)
            ref = torch.autograd.grad(obj, list(leaves.values()), retain_graph=True, allow_unused=True)
            for k, r in zip(leaves, ref):
                r = torch.zeros_like(leaves[k]) if r is None else r
                assert rel_err(grads[i][k].numpy(), r.numpy()) < 1e-12, (i, k)


def test_vjp_with_the_loss_cotangents_reproduces_training_grads(weights_npz):
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R, training as TR
    cr = make_crystals(9, 1, 12, seed=5)
    with f64_default():
        W, fw = _weights(weights_npz)
        tabs = R.DiffusionTables.build(T, Z)
        torch.manual_seed(4)
        G, N = cr.num_crystals, cr.total_atoms
        timestep, eps_x, u, eps_l = TR.draw_training_noise(G, N, Z, T)
        na, A0 = torch.as_tensor(cr.num_atoms), torch.as_tensor(cr.types)
        L0 = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles))
        loss, grads, p = TR.training_grads(W, tabs, fw, torch.as_tensor(cr.frac), A0, L0, na, timestep, eps_x, u, eps_l,
                                           5.0, 8)
        t_atom = timestep.reshape(-1).repeat_interleave(na)
        s, l, n = [p[k].clone().requires_grad_(True) for k in ("pred_eps", "pred_logits", "pred_len")]
        total = (TR.frac_x_error(s, p["target_eps"]) + TR.d3pm_calculate_loss(tabs, A0, l, p["noisy_types"], t_atom)[0]
                 + torch.nn.functional.mse_loss(n, p["lengths"] / na.unsqueeze(-1)))
        assert abs(total.item() - loss.item()) <= 1e-13 * abs(loss.item())
        cot = torch.autograd.grad(total, [s, l, n])
        outs, vjp, _ = TR.ponita_vjp(W, tabs, fw, p["noisy_frac"], p["noisy_types"], t_atom, na, p["noisy_lengths"],
                                     p["angles"], 5.0, 8, [cot], slice_crystals=4)
    assert rel_err(outs["score"].numpy(), p["pred_eps"].numpy()) < 1e-12
    assert rel_err(outs["logits"].numpy(), p["pred_logits"].numpy()) < 1e-12
    assert rel_err(outs["len0"].numpy(), p["pred_len"].numpy()) < 1e-12
    for k, g in grads.items():
        assert rel_err(vjp[0][k].numpy(), g.numpy()) < 1e-12, k


def test_gradient_blocks_partition_every_parameter(weights_npz):
    """Every element of every parameter lies in exactly one block, and the read-out blocks hold the rows they name."""
    from oracle import training as TR
    shapes = {k: weights_npz[k].shape for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    blocks = TR.gradient_blocks(shapes, Z, F)
    count = {k: np.zeros(s, dtype=np.int64) for k, s in shapes.items()}
    for _, parts in blocks:
        for k, idx in parts:
            count[k][idx] += 1
    for k, c in count.items():
        assert c.size and (c == 1).all(), k
    names = [b for b, _ in blocks]
    assert len(set(names)) == len(names)
    layers = sum(k.startswith("read_out_layers.") and k.endswith(".weight") for k in shapes)
    assert layers == 5 and len(blocks) == len(shapes) - 2 * layers + 3 * layers + 1
    by_name = dict(blocks)
    probe = {k: np.arange(int(np.prod(s))).reshape(s) for k, s in shapes.items()}
    (w, wi), (b, bi) = by_name["read_out_layers.2[score]"]
    assert probe[w][wi].shape == (1, 128) and probe[b][bi].tolist() == [Z]
    (w, wi), (b, bi) = by_name["read_out_layers.0[len0]"]
    assert probe[b][bi].tolist() == [Z + 1, Z + 2, Z + 3]
    (k, idx), = by_name["x_embedder.weight[vector]"]
    assert probe[k][idx].shape == (128, shapes[k][1] - F) and shapes[k][1] - F == 4
