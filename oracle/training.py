"""CPU restatement of Arreau's TRAINING step (SURVEY 8a rows a19-a23) -- TEST INFRASTRUCTURE ONLY.

Companion of oracle/restatement.py (same rules: only tests/, __graft_entry__.smoke() and bench.py's CPU legs
may import it).  It restates DiffusionLoss.__call__ (diffusion/diffusion_loss.py:204-274) and what it calls with
the random draws INJECTED (timestep per crystal, eps_x, u_type, eps_len -- in the reference's draw order, see
`draw_training_noise`), and obtains the parameter gradients with torch autograd on the restated forward
(oracle/restatement.py: ponita_forward), like the reference's `loss.backward()`.

`ponita_vjp` gives the network's parameter gradients for arbitrary output cotangents, computed crystal slice by
crystal slice, so that each output's share of the backward can be checked on its own and at full batch size.

Pinning: oracle/gen_golden.py::gen_training runs the LIVE reference's DiffusionLoss.__call__ + backward on the
same seeded batch, asserts this restatement equal (loss <= 1e-12, grads <= 1e-9 relative) and writes
tests/golden/train_c5small.npz.
"""
from __future__ import annotations

from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import torch

from . import restatement as R

HYBRID_LOSS_COEFF = 0.001   # diffusion/d3pm.py:15


# --------------------------------------------------------------------------------------
# forward noising
# --------------------------------------------------------------------------------------
def draw_training_noise(G: int, N: int, Z: int, T: int, generator=None):
    """The reference's draw order inside DiffusionLoss.__call__ (diffusion_loss.py:214-237): randint timestep
    [G,1]; VE_pbc.forward randn_like(frac) (helpers:45); D3PM.get_xt rand((N,Z)) (d3pm.py:141);
    VP_lattice.forward randn_like(lengths) (helpers:158)."""
    timestep = torch.randint(1, T + 1, size=(G, 1), generator=generator).long()
    eps_x = torch.randn(N, 3, generator=generator)
    u = torch.rand(N, Z, generator=generator)
    eps_l = torch.randn(G, 3, generator=generator)
    return timestep, eps_x, u, eps_l


def cart_to_frac_coords(cart: torch.Tensor, lattice: torch.Tensor, num_atoms: torch.Tensor) -> torch.Tensor:
    """diffusion/diffusion_helpers.py:233-251 (pinv of the lattice, then % 1)."""
    inv = torch.linalg.pinv(lattice)
    inv_nodes = torch.repeat_interleave(inv, num_atoms, dim=0)
    return torch.einsum("bi,bij->bj", cart, inv_nodes) % 1.0


def min_distance_vector_pbc(pos1: torch.Tensor, pos2: torch.Tensor, lattice: torch.Tensor, num_atoms: torch.Tensor):
    """diffusion/diffusion_helpers.py:254-325 with return_vector=True: over the 27 cells k (SUPERCELLS order),
    v_k = pos1 - (pos2 + c_k @ Lat); returns the v_k of least squared norm (first minimum wins, torch.min)."""
    cells = torch.tensor(R.SUPERCELLS, dtype=pos1.dtype)                    # [27,3]
    unit_cell = cells.T                                                      # [3,27]
    offs = torch.bmm(lattice.transpose(1, 2), unit_cell[None].expand(lattice.shape[0], -1, -1))   # [G,3,27]
    offs_atom = torch.repeat_interleave(offs, num_atoms, dim=0)
    v = pos1[:, :, None] - (pos2[:, :, None] + offs_atom)                    # [N,3,27]
    d2 = (v ** 2).sum(1)
    _, idx = d2.min(dim=-1)
    return torch.gather(v, 2, idx[:, None, None].repeat(1, 3, 1)).squeeze(-1)


def ve_pbc_forward(tabs: R.DiffusionTables, frac0, t_feat, lattice, num_atoms, eps):
    """diffusion/diffusion_helpers.py:43-63.  eps = the injected randn_like(frac0)."""
    sig = tabs.ve_sigmas[t_feat].view(-1, 1)
    frac_noisy = (frac0 + eps * sig) % 1
    cart_noisy = R.frac_to_cart_coords(frac_noisy, lattice, num_atoms)
    cart_p = R.frac_to_cart_coords(frac0, lattice, num_atoms)
    vec = min_distance_vector_pbc(cart_noisy, cart_p, lattice, num_atoms)
    return frac_noisy, cart_to_frac_coords(vec, lattice, num_atoms), sig


def vp_lattice_forward(tabs: R.DiffusionTables, h0, t, eps):
    """diffusion/diffusion_helpers.py:156-163; alpha_bars is fp32 (quirk B1), t is [G,1]."""
    ab = tabs.vp_alpha_bars[t]
    return torch.sqrt(ab).view(-1, 1) * h0 + torch.sqrt(1 - ab).view(-1, 1) * eps


def d3pm_q_sample(tabs: R.DiffusionTables, x0, t, u):
    """diffusion/d3pm.py:119-127."""
    logits = torch.log(tabs.q_mats[t - 1, x0, :] + R.D3PM_EPS)
    noise = torch.clip(u, R.D3PM_EPS, 1.0)
    return torch.argmax(logits - torch.log(-torch.log(noise)), dim=-1)


# --------------------------------------------------------------------------------------
# losses
# --------------------------------------------------------------------------------------
def frac_x_error(pred, target):
    """diffusion/diffusion_loss.py:95-110."""
    d = torch.clamp(torch.remainder((pred - target).abs(), 1), min=0, max=1)
    d = torch.min(d, 1 - d)
    return torch.mean(torch.sum(d ** 2, dim=1))


def d3pm_posterior_logits_from_int(tabs: R.DiffusionTables, x0, x_t, t):
    """diffusion/d3pm.py:74-110, integer x_0 branch (:81-84)."""
    logits = torch.log(torch.nn.functional.one_hot(x0, tabs.Z) + R.D3PM_EPS)
    return R.d3pm_q_posterior_logits(tabs, logits, x_t, t)


def d3pm_vb(dist1, dist2):
    """diffusion/d3pm.py:112-117."""
    out = torch.softmax(dist1 + R.D3PM_EPS, dim=-1) * (torch.log_softmax(dist1 + R.D3PM_EPS, dim=-1)
                                                        - torch.log_softmax(dist2 + R.D3PM_EPS, dim=-1))
    return out.sum(dim=-1).mean()


def d3pm_calculate_loss(tabs: R.DiffusionTables, x0, pred_logits, x_t, t):
    """diffusion/d3pm.py:145-163."""
    true_post = d3pm_posterior_logits_from_int(tabs, x0, x_t, t)
    pred_post = R.d3pm_q_posterior_logits(tabs, pred_logits, x_t, t)
    vb = d3pm_vb(true_post, pred_post)
    ce = torch.nn.functional.cross_entropy(pred_logits, x0)
    return vb * HYBRID_LOSS_COEFF + ce, vb, ce


# --------------------------------------------------------------------------------------
# the training step
# --------------------------------------------------------------------------------------
def training_loss(w: R.PonitaWeights, tabs: R.DiffusionTables, fourier_w, X0, A0, L0, num_atoms, timestep, eps_x, u,
                  eps_l, radius: float, max_neighbors: int, return_parts: bool = False):
    """DiffusionLoss.__call__ (diffusion/diffusion_loss.py:204-274) with the draws injected.
    X0[N,3] frac, A0[N] long, L0[G,3,3], num_atoms[G], timestep[G,1] long."""
    t_feat = timestep.repeat_interleave(num_atoms, dim=0)                     # [N,1]
    noisy_frac, target_eps, _sig = ve_pbc_forward(tabs, X0, t_feat, L0, num_atoms, eps_x)
    t_atom = t_feat.squeeze(-1)
    noisy_types = d3pm_q_sample(tabs, A0, t_atom, u)
    lengths, angles = R.matrix_to_params(L0)
    noisy_lengths = vp_lattice_forward(tabs, lengths, timestep, eps_l)
    onehot = torch.nn.functional.one_hot(noisy_types, tabs.Z)
    pred_eps, pred_logits, pred_len = R.predict_scores(w, tabs, fourier_w, noisy_frac, onehot, t_atom, num_atoms,
                                                       noisy_lengths, angles, radius, max_neighbors)
    e_frac = frac_x_error(pred_eps, target_eps)
    e_type, vb, ce = d3pm_calculate_loss(tabs, A0, pred_logits, noisy_types, t_atom)
    target_len = lengths / num_atoms.unsqueeze(-1)
    e_lat = torch.nn.functional.mse_loss(pred_len, target_len)
    loss = e_frac + e_type + e_lat
    if return_parts:
        parts = dict(noisy_frac=noisy_frac, target_eps=target_eps, noisy_types=noisy_types, lengths=lengths,
                     angles=angles, noisy_lengths=noisy_lengths, pred_eps=pred_eps, pred_logits=pred_logits,
                     pred_len=pred_len, e_frac=e_frac, e_type=e_type, vb=vb, ce=ce, e_lat=e_lat)
        return loss, parts
    return loss


def training_grads(w: R.PonitaWeights, *args, **kw) -> Tuple[torch.Tensor, Dict[str, torch.Tensor], dict]:
    """loss, {param name: dloss/dparam} (autograd on the restated forward = the reference's loss.backward()),
    and the intermediate parts."""
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in w.sd.items()}
    w2 = R.PonitaWeights(leaves, w.ori_grid, w.radius, w.num_layers)
    loss, parts = training_loss(w2, *args, return_parts=True, **kw)
    names = list(leaves)
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    g = {k: (torch.zeros_like(leaves[k]) if gv is None else gv) for k, gv in zip(names, grads)}
    return loss.detach(), g, {k: (v.detach() if isinstance(v, torch.Tensor) else v) for k, v in parts.items()}


def ponita_vjp(w: R.PonitaWeights, tabs: R.DiffusionTables, fourier_w, frac, types, t_atom, num_atoms, lengths, angles,
               radius: float, max_neighbors: int, cotangents: Sequence[Tuple[Optional[torch.Tensor], ...]],
               slice_crystals: Optional[int] = None, lattice: Optional[torch.Tensor] = None):
    """Vector-Jacobian products of R.predict_scores at one noised state: for every cotangent set (dscore[N,3],
    dlogits[N,Z], dlen0[G,3]; None = zero) the parameter gradients of <dscore, score> + <dlogits, logits> +
    <dlen0, len0>, i.e. autograd with those grad_outputs.  frac[N,3], types[N] (states, one-hot encoded here),
    t_atom[N], num_atoms[G], lengths / angles [G,3]; lattice [G,3,3] as in R.predict_scores.

    Computed as a sum over slices of `slice_crystals` whole crystals (default: the whole batch in one slice), one
    forward per slice and one backward per cotangent set.  This is exact, not an approximation: no edge crosses a
    crystal and every pooling is per crystal, so each slice is a batch of its own and the gradient of the batch is the
    sum of the slices' gradients.

    Returns (outputs {score, logits, len0} of the whole batch, [{param name: gradient}] per cotangent set, the graph:
    edge_index [2,E] with global atom indices (row 0 sender, row 1 receiver) and cell_offsets [E,3])."""
    num_atoms = torch.as_tensor(num_atoms, dtype=torch.long)
    G = int(num_atoms.shape[0])
    off = [0] + torch.cumsum(num_atoms, 0).tolist()
    step = G if slice_crystals is None else max(1, int(slice_crystals))
    onehot = torch.nn.functional.one_hot(torch.as_tensor(types, dtype=torch.long), tabs.Z).to(frac.dtype)
    t_atom = torch.as_tensor(t_atom, dtype=torch.long)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in w.sd.items()}
    w2 = R.PonitaWeights(leaves, w.ori_grid, w.radius, w.num_layers)
    names = list(leaves)
    grads = [{k: torch.zeros_like(leaves[k]) for k in names} for _ in cotangents]
    outs: Dict[str, list] = {"score": [], "logits": [], "len0": []}
    edges = []
    for g0 in range(0, G, step):
        g1 = min(G, g0 + step)
        a0, a1 = off[g0], off[g1]
        score, logits, len0, graph = R.predict_scores(w2, tabs, fourier_w, frac[a0:a1], onehot[a0:a1], t_atom[a0:a1],
                                                      num_atoms[g0:g1], lengths[g0:g1], angles[g0:g1], radius,
                                                      max_neighbors, return_graph=True,
                                                      lattice=None if lattice is None else lattice[g0:g1])
        edges.append((graph[0] + a0, graph[1]))
        for name, v in (("score", score), ("logits", logits), ("len0", len0)):
            outs[name].append(v.detach())
        for i, cot in enumerate(cotangents):
            pairs = [(y, c[rows]) for y, c, rows in zip((score, logits, len0), cot,
                                                        (slice(a0, a1), slice(a0, a1), slice(g0, g1))) if c is not None]
            if not pairs:
                continue
            gs = torch.autograd.grad([y for y, _ in pairs], [leaves[k] for k in names], [c.to(y.dtype) for y, c in pairs],
                                     retain_graph=i + 1 < len(cotangents), allow_unused=True)
            for k, gv in zip(names, gs):
                if gv is not None:
                    grads[i][k] += gv
    graph = ((torch.cat([e for e, _ in edges], 1), torch.cat([c for _, c in edges])) if edges else
             (torch.zeros(2, 0, dtype=torch.long), torch.zeros(0, 3, dtype=frac.dtype)))
    return {k: torch.cat(v) for k, v in outs.items()}, grads, graph


def gradient_blocks(shapes: Mapping[str, Sequence[int]], num_states: int, num_scalar: int
                    ) -> List[Tuple[str, List[Tuple[str, tuple]]]]:
    """A partition of every parameter element into the blocks a gradient is compared by: (block name, [(parameter
    name, index into that tensor)]).  Each read-out layer's weight and bias rows are split by the output they produce
    (logits rows [0, Z), the score row Z, the len0 rows Z+1..Z+3), a row's weight and bias in one block: the lattice
    term otherwise dominates the tensor and hides the others, and the score bias alone nearly cancels over the
    orientation grid.  x_embedder.weight is split into its scalar and its vector columns.  Every other tensor is one
    block."""
    Z, F = num_states, num_scalar
    blocks = []
    for k in shapes:
        if k.startswith("read_out_layers.") and k.endswith(".bias"):
            continue
        if k.startswith("read_out_layers.") and k.endswith(".weight"):
            kb = k[: -len("weight")] + "bias"
            for out, rows in (("logits", slice(0, Z)), ("score", slice(Z, Z + 1)), ("len0", slice(Z + 1, Z + 4))):
                blocks.append((f"{k[: -len('.weight')]}[{out}]", [(k, (rows, slice(None))), (kb, (rows,))]))
        elif k == "x_embedder.weight":
            blocks.append((k + "[scalar]", [(k, (slice(None), slice(0, F)))]))
            blocks.append((k + "[vector]", [(k, (slice(None), slice(F, None)))]))
        else:
            blocks.append((k, [(k, (Ellipsis,))]))
    return blocks


def calibrate(w: R.PonitaWeights, x, vec, edge_index, dists, direction, lattice, batch, num_graphs) -> Dict[str, torch.Tensor]:
    """FiberBundleConv.callibrate (ponita/nn/conv.py:122-123,140-146) as it acts during the FIRST train-mode
    forward: layer l rescales kernel.weight by std(x)/std(x1) and fiber_kernel.weight by std(x1)/std(x2), where
    x, x1, x2 are that forward's own tensors (computed with the weights BEFORE the rescale; later layers see the
    un-rescaled outputs of earlier ones).  Returns the new weights (a copy of the state dict)."""
    _, _, _, inter = R.ponita_forward(w, x, vec, edge_index, dists, direction, lattice, batch, num_graphs,
                                      out_dims=(w["read_out_layers.0.weight"].shape[0] - 4, 1, 0, 3),
                                      return_intermediates=True)
    out = dict(w.sd)
    h_in = inter["h0"]
    for l in range(w.num_layers):
        p = f"interaction_layers.{l}.conv."
        x1, x2 = inter[f"x1_{l}"], inter[f"x2_{l}"] - w[p + "bias"]         # std is taken before the bias is added
        out[p + "kernel.weight"] = w[p + "kernel.weight"] * (h_in.std() / x1.std())
        out[p + "fiber_kernel.weight"] = w[p + "fiber_kernel.weight"] * (x1.std() / x2.std())
        h_in = inter[f"h_{l}"]
    return out
