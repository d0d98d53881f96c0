"""Forward-only loss evaluation (validation / test loss) on the GPU.

Per batch: per-crystal keyed noise (arreau_eval_noise) -> upload -> the training step's noising
(`BatchEngine.noise_batch`) -> graph + forward (fp32 SIMT or fp16 tcgen05, the model's precision) -> per-crystal loss
sums (arreau_eval_loss).  No backward, no gradient buffers, no torch RNG: evaluation leaves the training run exactly as
it was.  Because every
crystal's draws are keyed by (seed, crystal id) and its loss terms are summed over its own atoms only, the per-crystal
numbers -- and every metric rebuilt from them -- do not depend on how the split is grouped into GPU batches or spread
over ranks.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import attr
import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .distributed import all_gather_rows, shard_range
from .training import HYBRID_LOSS_COEFF, BatchEngine

LOSS_PARTS = ("loss", "e_frac", "vb", "ce", "e_lat")


@attr.s(auto_attribs=True, frozen=True)
class EvalResult:
    """Per-crystal evaluation of one batch: t[G] i32 (device), num_atoms[G] i64 (host), terms[G,4] f64 (device) =
    {sum of the wrapped squared frac error, sum of vb, sum of ce over the crystal's atoms, sum_d (len0 - lengths/n)^2}."""
    t: torch.Tensor
    num_atoms: torch.Tensor
    terms: torch.Tensor


class EvalEngine(BatchEngine):
    """A capacity-sized DenoiseEngine (no debug buffers, no backward workspace) plus the noising buffers, re-bound per
    batch with `set_topology` like TrainEngine."""

    def _own_bufs(self, N: int, G: int, Z: int) -> Dict[str, tuple]:
        return {"crystal_ids": ("G", torch.zeros(G, dtype=torch.int64, device=self.device)),
                "per_crystal": ("G", torch.zeros(G, 4, dtype=torch.float64, device=self.device))}

    def run(self, frac0, types0, lattice0, crystal_ids, seed: int = 0, timestep=None, noise=None):
        """Loss terms per crystal of the bound batch; returns (t_crystal[G], per_crystal[G,4]) as views of the engine's
        buffers.  timestep (scalar or [G]) / noise (eps_x[N,3], u[N,Z], eps_l[G,3]) replace the keyed draws."""
        e, tb = self.eng, self.tabs
        ids = torch.as_tensor(crystal_ids, dtype=torch.int64).reshape(e.G)
        self.crystal_ids.copy_(ids.pin_memory() if ids.device.type == "cpu" else ids, non_blocking=True)
        if timestep is None or noise is None:
            _lib.call("arreau_eval_noise", C.c_uint64(int(seed)), e.G, e.N, e.Z, tb.T, self.crystal_ids.data_ptr(),
                      e.atom_offset.data_ptr(), e.crystal_of_atom.data_ptr(), self.t_crystal.data_ptr(),
                      self.eps_x.data_ptr(), self.u.data_ptr(), self.eps_l.data_ptr(), e.stream)
        self.upload_batch(frac0, types0, lattice0, timestep, noise)
        self.noise_batch()
        e.predict_scores(self.t_atom, from_trig=False)
        _lib.call("arreau_eval_loss", e.score.data_ptr(), e.logits.data_ptr(), e.len0.data_ptr(),
                  self.target_eps.data_ptr(), self.types0.data_ptr(), e.types.data_ptr(), self.t_atom.data_ptr(),
                  self.lengths0.data_ptr(), e.atom_offset.data_ptr(), e.d_q_keep.data_ptr(), e.d_q_to_mask.data_ptr(),
                  tb.onestep_keep, tb.onestep_to_mask, tb.T, e.N, e.G, e.Z, self.terms.data_ptr(),
                  self.per_crystal.data_ptr(), e.stream)
        return self.t_crystal, self.per_crystal


def batch_metric(num_atoms: np.ndarray, terms: np.ndarray, batch_size: int,
                 hybrid_coeff: float = HYBRID_LOSS_COEFF) -> Dict[str, float]:
    """The loss metric of `train.fit` over virtual batches of `batch_size` consecutive crystals: each batch's five
    scalars are rebuilt from the per-crystal sums with arreau_training_loss's formulas (frac, vb, ce / N_B, lattice
    / 3 G_B, loss = frac + (vb * coeff + ce) + lattice) and reduced like DiffusionLossMetric (sum over batches / number
    of crystals).  Returns {loss, e_frac, vb, ce, e_lat}."""
    num_atoms = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
    terms = np.asarray(terms, dtype=np.float64).reshape(-1, 4)
    n = num_atoms.shape[0]
    if n == 0:
        return {k: float("nan") for k in LOSS_PARTS}
    sums = [0.0] * 5
    for s in range(0, n, batch_size):
        tm, NB, GB = terms[s:s + batch_size], float(num_atoms[s:s + batch_size].sum()), min(batch_size, n - s)
        e_frac, vb, ce = tm[:, 0].sum() / NB, tm[:, 1].sum() / NB, tm[:, 2].sum() / NB
        e_lat = tm[:, 3].sum() / (3.0 * GB)
        for i, v in enumerate((e_frac + (vb * hybrid_coeff + ce) + e_lat, e_frac, vb, ce, e_lat)):
            sums[i] += float(v)
    return {k: v / n for k, v in zip(LOSS_PARTS, sums)}


@torch.no_grad()
def evaluate_dataset(model, dataset, batch_size: int, device, seed: int = 0, gpu_batch: Optional[int] = None) -> dict:
    """Loss of `model` on a split: {loss, e_frac, vb, ce, e_lat} (`batch_metric` over virtual batches of `batch_size`
    in dataset order, comparable with fit's train loss) and the per-crystal arrays crystal_ids, num_atoms, t, terms[n,4]
    in dataset order.  The split is evaluated `gpu_batch` crystals at a time (default `batch_size`); under DDP each rank
    evaluates a contiguous shard and the per-crystal terms are all-gathered once, so every rank returns the same
    result, independent of `gpu_batch` and of the world size.  With a capped graph the device is read once, at the end."""
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    device = torch.device(device)
    gpu_batch = int(gpu_batch or batch_size)
    n = len(dataset)
    ids = np.asarray(getattr(dataset, "crystal_ids", np.arange(n)), dtype=np.int64)
    counts = np.asarray(dataset.atom_counts(), dtype=np.int64)
    lo, hi = shard_range(n, rank, world)
    chunks = [np.arange(s, min(s + gpu_batch, hi)) for s in range(lo, hi, gpu_batch)]
    dl = model.diffusion_loss
    ts, terms = [], []
    if chunks:
        capacity = (max(int(counts[c].sum()) for c in chunks), max(len(c) for c in chunks))
        for c in chunks:
            batch = dataset.collate_indices(c, device=device)
            r = dl.evaluate(model, batch, model.t_emb, ids[c], seed=seed, capacity=capacity)
            ts.append(r.t)
            terms.append(r.terms)
        t_local, terms_local = torch.cat(ts).cpu().numpy(), torch.cat(terms).cpu().numpy()
    else:
        t_local, terms_local = np.zeros(0, dtype=np.int64), np.zeros((0, 4))
    comm = device if dist.is_initialized() and dist.get_backend() == "nccl" else None
    t_all, terms_all = all_gather_rows([t_local.astype(np.int64), terms_local], device=comm)
    out = batch_metric(counts, terms_all, batch_size)
    out.update(crystal_ids=ids, num_atoms=counts, t=t_all, terms=terms_all)
    return out
