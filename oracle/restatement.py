"""CPU restatement of Arreau's denoising step -- TEST INFRASTRUCTURE ONLY.

This file is the *oracle*: a plain-torch (CPU, fp64 by default) restatement of the
reference algorithm for the hot path (SURVEY.md section 8 / Appendix A).  It is NOT
part of the product: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import it.  The product (arreau_b200/) never imports oracle/.

Pinning: the reference ships no golden vectors (SURVEY.md section 4).  This restatement is
pinned against the LIVE reference (the unmodified files under /root/reference imported
with oracle/shims) by oracle/gen_golden.py, which also writes tests/golden/*.npz; the
`-m "not gpu"` tests re-check the restatement against those committed vectors.

Every function cites the reference file:line it restates (paths relative to the
reference root).  Run under torch.set_default_dtype(torch.float64) for reference parity
(the reference always runs fp64: main_diffusion_generate.py:27).
"""
from __future__ import annotations

import itertools
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

# diffusion/diffusion_helpers.py:10  -- cell k = k-th element of product((-1,0,1), repeat=3)
SUPERCELLS: List[Tuple[int, int, int]] = list(itertools.product((-1, 0, 1), repeat=3))

# diffusion/diffusion_loss.py:30-36
POS_SIGMA_MIN = 0.001
POS_SIGMA_MAX = 1.0
LATTICE_POWER = 2
LATTICE_CLIPMAX = 0.999
# lightning_wrappers/diffusion.py:22-23
FOURIER_SCALE = 16
T_EMB_DIM = 64
# diffusion/d3pm.py:23,34
D3PM_EPS = 1e-6
D3PM_MASK_RATE = 0.02


# --------------------------------------------------------------------------------------
# schedules (init-time tables)
# --------------------------------------------------------------------------------------
def ve_sigmas(T: int, sigma_min: float = POS_SIGMA_MIN, sigma_max: float = POS_SIGMA_MAX) -> torch.Tensor:
    """diffusion/diffusion_helpers.py:38-41 (VE_pbc.__init__): default-dtype linspace of logs."""
    return torch.exp(torch.linspace(np.log(sigma_min), np.log(sigma_max), T + 1))


def vp_schedule(T: int, s: float = 0.0001, power: int = LATTICE_POWER, clipmax: float = LATTICE_CLIPMAX):
    """diffusion/diffusion_helpers.py:141-154 (VP_lattice.__init__).

    Built in fp32 (`dtype=torch.float`), then `cat` with a default-dtype zero promotes
    betas/sigmas (alpha_bars stays fp32) -- quirk B1."""
    t = torch.arange(0, T + 1, dtype=torch.float)
    f_t = torch.cos((np.pi / 2) * ((t / T) + s) / (1 + s)) ** power
    alpha_bars = f_t / f_t[0]
    betas = torch.cat([torch.zeros([1]), 1 - (alpha_bars[1:] / alpha_bars[:-1])], dim=0)
    betas = betas.clamp_max(clipmax)
    sigmas = torch.sqrt(betas[1:] * ((1 - alpha_bars[:-1]) / (1 - alpha_bars[1:])))
    sigmas = torch.cat([torch.zeros([1]), sigmas], dim=0)
    return alpha_bars, betas, sigmas


def d3pm_mask_matrices(T: int, Z: int):
    """diffusion/d3pm.py:25-59: one-step (transposed) and cumulative mask-absorbing matrices."""
    mat = torch.zeros(Z, Z)
    mat[:, -1] = torch.full((Z,), D3PM_MASK_RATE)
    mat.diagonal().fill_(1 - D3PM_MASK_RATE)
    mat[-1, -1] = 1
    one_step = [mat.clone() for _ in range(T)]
    q_one_step_transposed = torch.stack(one_step, 0).transpose(1, 2)
    q = one_step[0]
    q_mats = [q]
    for idx in range(1, T):
        q = q @ one_step[idx]
        q_mats.append(q)
    return q_one_step_transposed, torch.stack(q_mats, 0)


# --------------------------------------------------------------------------------------
# lattice / coordinates
# --------------------------------------------------------------------------------------
def lattice_from_params(lengths: torch.Tensor, angles: torch.Tensor) -> torch.Tensor:
    """diffusion/lattice_helpers.py:55-105 (angles are consumed as radians)."""
    a, b, c = lengths.unbind(-1)
    alpha, beta, gamma = angles.unbind(-1)
    cos_a, cos_b, cos_g = torch.cos(alpha), torch.cos(beta), torch.cos(gamma)
    sin_a, sin_b = torch.sin(alpha), torch.sin(beta)
    val = torch.clamp((cos_a * cos_b - cos_g) / (sin_a * sin_b), -1.0, 1.0)
    gamma_star = torch.arccos(val)
    zero = torch.zeros_like(a)
    va = torch.stack([a * sin_b, zero, a * cos_b], dim=1)
    vb = torch.stack([-b * sin_a * torch.cos(gamma_star), b * sin_a * torch.sin(gamma_star), b * cos_a], dim=1)
    vc = torch.stack([zero, zero, c], dim=1)
    return torch.cat([va, vb, vc], dim=-1).view(-1, 3, 3)


def matrix_to_params(matrix: torch.Tensor):
    """diffusion/lattice_helpers.py:16-35."""
    lengths = torch.sqrt(torch.sum(matrix ** 2, dim=-1))
    angles = torch.zeros((matrix.shape[0], 3), dtype=matrix.dtype)
    for i in range(3):
        j, k = (i + 1) % 3, (i + 2) % 3
        angles[..., i] = torch.acos(torch.clamp(
            torch.sum(matrix[..., j, :] * matrix[..., k, :], dim=-1) / (lengths[..., j] * lengths[..., k]),
            -1.0, 1.0))
    return lengths, angles


def frac_to_cart_coords(frac: torch.Tensor, lattice: torch.Tensor, num_atoms: torch.Tensor) -> torch.Tensor:
    """diffusion/diffusion_helpers.py:223-230."""
    lat_nodes = torch.repeat_interleave(lattice, num_atoms, dim=0)
    return torch.einsum("bi,bij->bj", frac, lat_nodes)


def fourier_time_embedding(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """diffusion/diffusion_helpers.py:23-25 (GaussianFourierProjection.forward)."""
    x_proj = x * w[None, :] * 2 * np.pi
    return torch.cat([torch.sin(x_proj), torch.cos(x_proj)], dim=-1)


# --------------------------------------------------------------------------------------
# periodic radius graph
# --------------------------------------------------------------------------------------
def radius_graph_pbc(cart: torch.Tensor, lattice: torch.Tensor, num_atoms: torch.Tensor, radius: float,
                     max_neighbors: int, remove_self_edges: bool = True):
    """diffusion/diffusion_helpers.py:328-564, restated per crystal.

    For every crystal g, receiver i, sender j (all n_g^2 pairs, j == i included) and cell
    k in 0..26: off = c_k @ Lat_g (:392-393), dir = (pos_j + off) - pos_i (:404,408),
    d2 = dx^2 + dy^2 + dz^2 (:409); keep d2 <= r^2 and d2 > 1e-4 (:432-436).  If the cap is
    positive, every receiver keeps its `cap` nearest (:469-536; a no-op for receivers at or
    below the cap, so the reference's global `max > cap` switch needs no special case).
    Exact d2 ties are broken by ascending (j, k) == torch.sort(stable=True) -- the build's
    canonical rule (SURVEY Appendix B4; the reference's own tie order is implementation
    defined).  Output order is (i, j, k) ascending.

    Returns (edge_index[2,E] int64 with row0 = sender j, row1 = receiver i,
             cell_offsets[E,3] = -cell, num_neighbors_image[G], dist[E], dir[E,3]).
    """
    dt = cart.dtype
    cells = torch.tensor(SUPERCELLS, dtype=dt)                                  # [27,3]
    r2 = radius * radius
    src_l, dst_l, cell_l, d2_l, dir_l, nimg = [], [], [], [], [], []
    start = 0
    for g, n in enumerate(num_atoms.tolist()):
        pos = cart[start:start + n]
        # bmm(lattice^T, cells^T): off[a,k] = sum_m Lat[m,a] * c_k[m]           (:390-393)
        # (products with c in {-1,0,1} are exact; the additions run m = 0,1,2 in order, which is
        # what the reference's CPU bmm does bit for bit -- checked by oracle/gen_golden.py)
        L = lattice[g]
        off = (cells[:, 0:1] * L[0][None, :] + cells[:, 1:2] * L[1][None, :]) + cells[:, 2:3] * L[2][None, :]  # [27,3]
        # dir[i,j,k,:] = (pos_j + off_k) - pos_i
        d = (pos[None, :, None, :] + off[None, None, :, :]) - pos[:, None, None, :]
        d2 = (d[..., 0] ** 2 + d[..., 1] ** 2) + d[..., 2] ** 2                   # [n,n,27], x,y,z in order
        mask = d2 <= r2
        if remove_self_edges:
            mask = mask & (d2 > 0.0001)
        # num_neighbors_image = sum_i min(count_i, cap) from the PRE-cap counts, also when the cap
        # is disabled (cap <= 0 -> zeros / negatives): helpers:456-465, a quirk kept as is.
        counts = mask.view(n, -1).sum(1)
        nimg.append(int(torch.clamp(counts, max=max_neighbors).sum()))
        if max_neighbors > 0:
            flat_d2 = torch.where(mask, d2, torch.full_like(d2, float("inf"))).view(n, n * 27)
            order = torch.sort(flat_d2, dim=1, stable=True)[1][:, :max_neighbors]
            keep = torch.zeros(n, n * 27, dtype=torch.bool)
            keep.scatter_(1, order, True)
            mask = mask & keep.view(n, n, 27)
        ii, jj, kk = torch.nonzero(mask, as_tuple=True)                         # (i, j, k) ascending
        src_l.append(jj + start)
        dst_l.append(ii + start)
        cell_l.append(cells[kk])
        d2_l.append(d2[ii, jj, kk])
        dir_l.append(d[ii, jj, kk])
        start += n
    if src_l:
        src, dst = torch.cat(src_l), torch.cat(dst_l)
        cell, d2c, dirc = torch.cat(cell_l), torch.cat(d2_l), torch.cat(dir_l)
    else:
        src = dst = torch.zeros(0, dtype=torch.long)
        cell = torch.zeros(0, 3, dtype=dt); d2c = torch.zeros(0, dtype=dt); dirc = torch.zeros(0, 3, dtype=dt)
    return (torch.stack((src, dst)), -cell, torch.tensor(nimg, dtype=torch.long),
            torch.sqrt(d2c), dirc)


# --------------------------------------------------------------------------------------
# Ponita fiber-bundle forward
# --------------------------------------------------------------------------------------
def polynomial_features(x: torch.Tensor, degree: int = 3) -> torch.Tensor:
    """ponita/nn/embedding.py:10-14: [x, x(x)x, (x(x)x)(x)x] flattened (258 for 6 inputs)."""
    out = [x]
    for _ in range(1, degree):
        out.append(torch.einsum("...i,...j->...ij", out[-1], x).flatten(-2, -1))
    return torch.cat(out, -1)


def polynomial_cutoff(x: torch.Tensor, r_max: float, p: float = 6.0) -> torch.Tensor:
    """ponita/utils/windowing.py:21-29."""
    env = (1.0 - ((p + 1.0) * (p + 2.0) / 2.0) * torch.pow(x / r_max, p)
           + p * (p + 2.0) * torch.pow(x / r_max, p + 1)
           - (p * (p + 1.0) / 2) * torch.pow(x / r_max, p + 2))
    return env * (x < r_max)


def gelu(x: torch.Tensor) -> torch.Tensor:
    """torch.nn.GELU() exact erf form (ponita/models/ponita.py:61)."""
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _cosine_similarity(a: torch.Tensor, b: torch.Tensor, eps: float = 1e-8) -> torch.Tensor:
    """torch.nn.CosineSimilarity(dim=-1) (ponita/transforms/invariants.py:27,83-85):
    torch computes x.y / sqrt(clamp(|x|^2 |y|^2, eps^2))."""
    w12 = (a * b).sum(-1)
    w1 = (a * a).sum(-1)
    w2 = (b * b).sum(-1)
    return w12 / torch.sqrt(torch.clamp(w1 * w2, min=eps * eps))


@dataclass
class PonitaWeights:
    """Plain tensors keyed like the reference state_dict (SURVEY 8b), plus the orientation
    grid (not part of the state_dict, quirk B2)."""
    sd: Dict[str, torch.Tensor]
    ori_grid: torch.Tensor          # [O,3]
    radius: float
    num_layers: int = 5

    def __getitem__(self, k):
        return self.sd[k]


def ponita_forward(w: PonitaWeights, x: torch.Tensor, vec: torch.Tensor, edge_index: torch.Tensor,
                   dists: torch.Tensor, direction: torch.Tensor, lattice: torch.Tensor,
                   batch: torch.Tensor, num_graphs: int, out_dims=(90, 1, 0, 3),
                   return_intermediates: bool = False):
    """ponita/models/ponita.py:88-123 with the transforms and layers it calls.

    x[N,F] scalars, vec[N,V,3] vectors, edge_index[2,E] (row0 sender, row1 receiver),
    dists[E], direction[E,3] (= pos_j + off - pos_i), lattice[G,3,3], batch[N].
    """
    ori = w.ori_grid.to(x.dtype)
    O = ori.shape[0]
    N = x.shape[0]
    src, dst = edge_index[0], edge_index[1]
    inter: Dict[str, torch.Tensor] = {}

    # lift: ponita/transforms/position_orientation_graph.py:84-86, ponita/utils/to_from_sphere.py:4-8
    x_lift = torch.cat([x.unsqueeze(1).expand(-1, O, -1), torch.einsum("bcd,nd->bnc", vec, ori)], dim=-1)

    # edge invariants: ponita/geometry/invariants.py:17-22, ponita/transforms/invariants.py:81-87
    rel = direction[:, None, :]
    inv1 = (rel * ori[None]).sum(-1, keepdim=True)
    inv2 = (rel - inv1 * ori[None]).norm(dim=-1, keepdim=True)
    fiber_attr = (ori[None, :, :] * ori[:, None, :]).sum(-1, keepdim=True)          # [O,O,1]
    lat_e = lattice[batch[src]]
    cs = [_cosine_similarity(direction, lat_e[:, m, :]) for m in range(3)]
    edge_scalar = torch.stack([dists, cs[0], cs[1], cs[2]], dim=-1)                 # [E,4]
    attr = torch.cat([inv1, inv2, edge_scalar[:, None, :].expand(-1, O, -1)], dim=-1)  # [E,O,6]

    # kernel bases: ponita/models/ponita.py:65-67,94-95
    def mlp(prefix, a):
        h = polynomial_features(a, 3)
        h = gelu(h @ w[prefix + ".1.weight"].T + w[prefix + ".1.bias"])
        return gelu(h @ w[prefix + ".3.weight"].T + w[prefix + ".3.bias"])

    kernel_basis = mlp("basis_fn", attr) * polynomial_cutoff(dists, w.radius)[:, None, None]  # [E,O,D]
    fiber_kernel_basis = mlp("fiber_basis_fn", fiber_attr)                                     # [O,O,D]

    h = x_lift @ w["x_embedder.weight"].T                                           # ponita.py:98
    if return_intermediates:
        inter["attr"] = attr; inter["kernel_basis"] = kernel_basis; inter["h0"] = h

    readouts = []
    for l in range(w.num_layers):
        p = f"interaction_layers.{l}."
        # ponita/nn/conv.py:110-111,131-133 + PyG add-aggregation
        kernel = kernel_basis @ w[p + "conv.kernel.weight"].T                        # [E,O,C]
        msg = kernel * h[src]
        x1 = torch.zeros_like(h).index_add_(0, dst, msg)
        # conv.py:113-115,126-127
        fk = fiber_kernel_basis @ w[p + "conv.fiber_kernel.weight"].T                # [O,O,C]
        x2 = torch.einsum("boc,opc->bpc", x1, fk) / O + w[p + "conv.bias"]
        # ponita/nn/convnext.py:25-32
        y = torch.nn.functional.layer_norm(x2, (x2.shape[-1],), w[p + "norm.weight"], w[p + "norm.bias"], 1e-5)
        y = gelu(y @ w[p + "linear_1.weight"].T + w[p + "linear_1.bias"])
        y = y @ w[p + "linear_2.weight"].T + w[p + "linear_2.bias"]
        h = w[p + "layer_scale"] * y + h
        readouts.append(h @ w[f"read_out_layers.{l}.weight"].T + w[f"read_out_layers.{l}.bias"])  # ponita.py:105
        if return_intermediates:
            inter[f"x1_{l}"] = x1; inter[f"x2_{l}"] = x2; inter[f"h_{l}"] = h

    readout = sum(readouts) / len(readouts)                                          # ponita.py:108
    d_s, d_v, d_gv, d_gs = out_dims
    r_s, r_v, _r_gv, r_gs = torch.split(readout, [d_s, d_v, d_gv, d_gs], dim=-1)     # ponita.py:111
    out_scalar = r_s.mean(dim=-2)                                                    # to_from_sphere.py:13-14
    out_vec = torch.einsum("bnc,nd->bcd", r_v, ori) / O                              # to_from_sphere.py:10-11
    gs = r_gs.mean(dim=-2)
    out_global = torch.zeros(num_graphs, d_gs, dtype=x.dtype).index_add_(0, batch, gs)  # ponita.py:152
    if return_intermediates:
        return out_scalar, out_vec, out_global, inter
    return out_scalar, out_vec, out_global


# --------------------------------------------------------------------------------------
# the step
# --------------------------------------------------------------------------------------
@dataclass
class DiffusionTables:
    """Init-time tables of DiffusionLoss (diffusion/diffusion_loss.py:68-93)."""
    T: int
    Z: int
    ve_sigmas: torch.Tensor
    vp_alpha_bars: torch.Tensor
    vp_betas: torch.Tensor
    vp_sigmas: torch.Tensor
    q_one_step_transposed: torch.Tensor
    q_mats: torch.Tensor

    @staticmethod
    def build(T: int, Z: int) -> "DiffusionTables":
        ab, b, s = vp_schedule(T)
        q1t, qm = d3pm_mask_matrices(T, Z)
        return DiffusionTables(T, Z, ve_sigmas(T), ab, b, s, q1t, qm)


def predict_scores(w: PonitaWeights, tabs: DiffusionTables, fourier_w: torch.Tensor, frac: torch.Tensor,
                   types_onehot: torch.Tensor, t: torch.Tensor, num_atoms: torch.Tensor, lengths: torch.Tensor,
                   angles: torch.Tensor, radius: float, max_neighbors: int, return_graph: bool = False,
                   lattice: Optional[torch.Tensor] = None):
    """diffusion/diffusion_loss.py:112-197.  `lattice` [G,3,3], when given, replaces lattice_from_params(lengths,
    angles): a caller comparing with another implementation passes that implementation's lattice, because its sin/cos
    may differ in the last bit, and the mirror images of an atom are exactly as far away as each other, so which of
    such a pair the neighbour cap keeps is decided by that bit."""
    G = num_atoms.shape[0]
    lat = lattice_from_params(lengths, angles) if lattice is None else lattice
    tt = tabs.vp_betas[t].view(-1, 1)
    t_emb = fourier_time_embedding(tt, fourier_w)
    rep = lambda a: torch.repeat_interleave(a, num_atoms, dim=0)
    scalar_feats = torch.cat([types_onehot, t_emb, rep(num_atoms).unsqueeze(-1), rep(lengths), rep(angles),
                              rep((lengths / num_atoms.unsqueeze(-1)).abs())], dim=1)
    cart = frac_to_cart_coords(frac, lat, num_atoms)
    vec = torch.cat([frac.unsqueeze(1), rep(lat)], dim=1)
    batch = torch.repeat_interleave(torch.arange(G), num_atoms)
    ei, cell_off, nimg, dist, direction = radius_graph_pbc(cart, lat, num_atoms, radius, max_neighbors)
    logits, vecs, len0 = ponita_forward(w, scalar_feats, vec, ei, dist, direction, lat, batch, G,
                                        out_dims=(tabs.Z, 1, 0, 3))
    if return_graph:
        return vecs.squeeze(1), logits, len0, (ei, cell_off, nimg, dist, direction)
    return vecs.squeeze(1), logits, len0


def vp_lattice_reverse_given_x0(tabs: DiffusionTables, xt, pred_x0, t, z):
    """diffusion/diffusion_helpers.py:185-199; `variance * z` (not its sqrt) is quirk B5.
    t is a 1-element long tensor; z is the injected randn_like(xt)."""
    denominator = 1 - tabs.vp_alpha_bars[t]
    alpha_t = 1 - tabs.vp_betas[t]
    x0_term = torch.sqrt(tabs.vp_alpha_bars[t - 1]) * tabs.vp_betas[t] * pred_x0
    xt_term = torch.sqrt(alpha_t) * (1 - tabs.vp_alpha_bars[t - 1]) * xt
    mean = (x0_term + xt_term) / denominator
    variance = (1 - tabs.vp_alpha_bars[t - 1]) * tabs.vp_betas[t] / denominator
    zz = torch.where((t > 1)[:, None].expand_as(xt), z, torch.zeros_like(xt))
    return mean + variance * zz


def ve_pbc_reverse(tabs: DiffusionTables, xt, eps_x, t, z):
    """diffusion/diffusion_helpers.py:65-81; z is the injected randn_like(xt)."""
    sig = tabs.ve_sigmas[t].view(-1, 1)
    adj = torch.where((t == 0).view(-1, 1), torch.zeros_like(sig), tabs.ve_sigmas[t - 1].view(-1, 1))
    mean = xt - eps_x * (sig ** 2 - adj ** 2)
    rand = torch.sqrt((adj ** 2 * (sig ** 2 - adj ** 2)) / (sig ** 2)) * z
    return (mean + rand) % 1


def d3pm_q_posterior_logits(tabs: DiffusionTables, x0_logits, x_t, t):
    """diffusion/d3pm.py:74-110 (float-logit branch)."""
    fact1 = tabs.q_one_step_transposed[t - 1, x_t, :]
    softmaxed = torch.softmax(x0_logits, dim=-1)
    qmats2 = tabs.q_mats[t - 2]
    fact2 = torch.einsum("bc,bcd->bd", softmaxed, qmats2)
    out = torch.log(fact1 + D3PM_EPS) + torch.log(fact2 + D3PM_EPS)
    return torch.where((t == 1).view(-1, 1), x0_logits, out)


def d3pm_reverse(tabs: DiffusionTables, x_t, x0_logits, t, u):
    """diffusion/d3pm.py:198-215; u is the injected torch.rand((N, Z))."""
    lp = d3pm_q_posterior_logits(tabs, x0_logits, x_t, t)
    noise = torch.clip(u, D3PM_EPS, 1.0)
    nfs = 0.2 + (t != 1).to(u.dtype).view(-1, 1) * 0.8
    gumbel = -torch.log(-torch.log(noise))
    return torch.argmax(lp + gumbel * nfs, dim=-1)


def denoise_step(w: PonitaWeights, tabs: DiffusionTables, fourier_w, frac, types, lengths, angles, num_atoms,
                 timestep: int, z_len, z_frac, u_type, radius: float, max_neighbors: int):
    """One iteration of the sampler loop, diffusion/diffusion_loss.py:318-349.
    Returns (frac', types', lengths', lattice', score, logits, len0)."""
    N = frac.shape[0]
    t = torch.full((N,), timestep, dtype=torch.long)
    tv = torch.tensor([timestep])
    onehot = torch.nn.functional.one_hot(types, tabs.Z)
    score, logits, len0 = predict_scores(w, tabs, fourier_w, frac, onehot, t, num_atoms, lengths, angles,
                                         radius, max_neighbors)
    pred_scaled = len0 * num_atoms.unsqueeze(-1)
    lengths_n = vp_lattice_reverse_given_x0(tabs, lengths, pred_scaled, tv, z_len)
    lattice_n = lattice_from_params(lengths_n, angles)
    frac_n = ve_pbc_reverse(tabs, frac, score, t, z_frac)
    types_n = d3pm_reverse(tabs, types, logits, t, u_type)
    return frac_n, types_n, lengths_n, lattice_n, score, logits, len0
