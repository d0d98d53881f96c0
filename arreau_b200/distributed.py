"""Box-level sharding of independent crystals (SURVEY 8e): one process per GPU, contiguous blocks of crystals
per rank, whole trajectories per GPU, and ONE collective at the end (gather of the sampled crystals).  There is
no per-step communication: graph edges never cross crystals (diffusion_helpers.py:350-383)."""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .diffusion.diffusion_loss import SampleResult


def shard_range(num_crystals: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous [lo, hi) block of crystals owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(num_crystals, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_rows(arrays: Sequence[np.ndarray], group=None, device: Optional[torch.device] = None) -> List[np.ndarray]:
    """All-gather arrays that are ragged in their leading dimension (each array its own row count per rank) and
    concatenate every array's parts in rank order.  Floating arrays travel as float64, integer arrays as int64.
    Counts first (one collective), then one padded payload per array.  Uses the group's backend (NCCL on the GPUs,
    gloo in the CPU tests); world size 1 returns the arrays unchanged."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return list(arrays)
    world = dist.get_world_size(group)
    dev = device if device is not None else torch.device("cpu")
    n_rows = torch.tensor([a.shape[0] for a in arrays], dtype=torch.int64, device=dev)
    counts = [torch.zeros_like(n_rows) for _ in range(world)]
    dist.all_gather(counts, n_rows, group=group)
    counts = torch.stack(counts).cpu().numpy()
    out = []
    for i, arr in enumerate(arrays):
        dtype = torch.float64 if np.asarray(arr).dtype.kind == "f" else torch.int64
        t = torch.zeros((int(counts[:, i].max()),) + arr.shape[1:], dtype=dtype, device=dev)
        t[: arr.shape[0]] = torch.as_tensor(arr, dtype=dtype)
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        out.append(np.concatenate([p[: int(counts[r, i])].cpu().numpy() for r, p in enumerate(parts)]))
    return out


def gather_crystal_metrics(local, group=None, device: Optional[torch.device] = None):
    """All-gather every rank's per-crystal CrystalMetrics rows (inference/crystal_metrics.py) into the whole set, in
    rank order -- one all_gather_rows.  A collective: every rank joins, also one with no crystals."""
    from .inference.crystal_metrics import METRIC_FIELDS, metrics_from_rows
    return metrics_from_rows(all_gather_rows([np.asarray(getattr(local, k)) for k in METRIC_FIELDS], group, device))


def gather_rng_states(state: torch.Tensor, group=None, device: Optional[torch.device] = None) -> List[torch.Tensor]:
    """Every rank's generator state (a uint8 tensor such as torch.cuda.get_rng_state() returns) in rank order, on every
    rank.  A collective (all_gather_rows): every rank must join it.  World size 1: [state]."""
    rows = all_gather_rows([state.cpu().numpy().astype(np.int64).reshape(1, -1)], group, device)[0]
    return [torch.as_tensor(r.astype(np.uint8)) for r in rows]


def rank_rng_state(states: Sequence[torch.Tensor], group=None) -> torch.Tensor:
    """This rank's entry of a `gather_rng_states` list written at the same world size."""
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if len(states) != world:
        raise ValueError(f"generator states of {len(states)} ranks cannot be restored at world size {world}")
    return torch.as_tensor(states[rank], dtype=torch.uint8)


def gather_sample_results(local: SampleResult, group=None, device: Optional[torch.device] = None) -> SampleResult:
    """All-gather the per-rank SampleResult (ragged in atoms) into the global one, rank-major = crystal order."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local
    frac, zs, lat, num_atoms = all_gather_rows([np.asarray(local.frac_x, dtype=np.float64),
                                                np.asarray(local.atomic_numbers, dtype=np.int64),
                                                np.asarray(local.lattice, dtype=np.float64),
                                                np.asarray(local.num_atoms, dtype=np.int64)], group, device)
    idx_start = np.concatenate([[0], np.cumsum(num_atoms)[:-1]]) if num_atoms.size else num_atoms
    return SampleResult(frac_x=frac, atomic_numbers=zs, lattice=lat, idx_start=idx_start, num_atoms=num_atoms)


def allreduce_gradients(flat_grad: torch.Tensor, group=None) -> torch.Tensor:
    """The DDP step of the training config (SURVEY 8e, C5): ONE all-reduce of the flat gradient buffer
    (1 170 646 fp32 = 4.7 MB), averaged over the ranks like Lightning's DDP strategy.  NCCL on the GPUs, gloo in
    the CPU tests.  In place; returns the buffer."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM, group=group)
        flat_grad.div_(dist.get_world_size(group))
    return flat_grad


def reduce_loss_metric(total_loss: torch.Tensor, total_samples: torch.Tensor, group=None) -> torch.Tensor:
    """DiffusionLossMetric (diffusion/diffusion_loss.py:52-65): both states are summed over the ranks
    (dist_reduce_fx="sum"), compute() = total_loss / total_samples."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        pair = torch.stack([total_loss.double().reshape(()), total_samples.double().reshape(())])
        dist.all_reduce(pair, op=dist.ReduceOp.SUM, group=group)
        return pair[0] / pair[1]
    return total_loss.double() / total_samples.double()


def broadcast_parameters(flat_data: torch.Tensor, src: int = 0, group=None) -> torch.Tensor:
    """Replicas start from rank `src`'s weights (DDP's initial broadcast)."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(flat_data, src=src, group=group)
    return flat_data
