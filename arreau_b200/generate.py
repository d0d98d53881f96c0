"""Mirror of main_diffusion_generate.py:52-94 (generate_n_crystals) on the GPU(s).

    python -m arreau_b200.generate --model_path model.ckpt --num_crystals 1024 --num_atoms 40 [--batch 1024]
    python -m arreau_b200.generate --model_path model.ckpt --num_crystals 1024 --num_atoms_from data/train.h5
    python -m arreau_b200.generate ... --keyed_noise      # the same crystals whatever --batch and the number of GPUs
    torchrun --nproc-per-node 8 -m arreau_b200.generate ...      # crystals sharded over the GPUs, one gather at the end

The reference samples 10 crystals per batch on the CPU; here a batch is as large as fits (1024 by default), every
GPU runs whole trajectories of its own contiguous block of crystals (arreau_b200.distributed.shard_range) and the only
collective is the final gather.  Output: out/crystals.h5 layout (inference/process_generated_crystals.py)."""
from __future__ import annotations

import argparse
import os
import time
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from .diffusion.diffusion_loss import SampleResult
from .distributed import gather_sample_results, shard_range
from .inference.process_generated_crystals import save_sample_results_to_hdf5

OUT_DIR = "out"


def generate_n_crystals(model, num_crystals: int, num_atoms_per_sample: Optional[int],
                        use_constant_atomic_symbols: Optional[list] = None, num_crystals_per_batch: int = 1024,
                        device="cuda", device_noise: bool = True, seed: int = 0, out_path: Optional[str] = None,
                        group=None, timings: Optional[dict] = None, num_atoms=None,
                        keyed_noise: bool = False) -> SampleResult:
    """main_diffusion_generate.py:52-94.  With torch.distributed initialised the crystals are sharded over the ranks;
    every rank returns the full gathered result and rank 0 writes `out_path`.  `timings` (optional dict) receives this
    rank's wall-clock seconds per phase: `sample` (list, one per batch), `gather`, `write`.  `num_atoms` (optional,
    length num_crystals) gives every crystal its own atom count instead of `num_atoms_per_sample`; each rank samples
    its shard of it (see `draw_num_atoms`).  `keyed_noise`: crystal i of the run gets id i and every draw of its
    trajectory is keyed by (seed, i) on the device (DiffusionLoss.sample's crystal_ids), so the result does not depend
    on num_crystals_per_batch or on the number of ranks.  Without it, batch b0.. is sampled with seed + b0."""
    if num_atoms is not None:
        num_atoms = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
        if num_atoms.shape[0] != num_crystals or np.any(num_atoms < 1):
            raise ValueError(f"num_atoms must hold {num_crystals} positive counts, got {num_atoms.shape[0]}")
        if use_constant_atomic_symbols is not None:
            raise ValueError("constant atomic symbols fix the atom count: they cannot be combined with num_atoms")
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    lo, hi = shard_range(num_crystals, rank, world)
    parts = []
    t_batches = []
    for b0 in range(lo, hi, num_crystals_per_batch):
        nb = min(num_crystals_per_batch, hi - b0)
        kw = {} if num_atoms is None else {"num_atoms": torch.from_numpy(num_atoms[b0:b0 + nb].copy())}
        if keyed_noise:
            kw["crystal_ids"] = torch.arange(b0, b0 + nb, dtype=torch.int64)
        t0 = time.perf_counter()
        parts.append(model.sample(num_atoms_per_sample=num_atoms_per_sample, num_samples_in_batch=nb,
                                  use_constant_atomic_symbols=use_constant_atomic_symbols, device=device,
                                  device_noise=device_noise, seed=seed if keyed_noise else seed + b0, **kw))
        t_batches.append(time.perf_counter() - t0)      # sample() ends with the device->host copy of the result
    n_local = hi - lo
    if parts:
        na = np.full(n_local, num_atoms_per_sample, dtype=np.int64) if num_atoms is None else num_atoms[lo:hi].copy()
        local = SampleResult(frac_x=np.concatenate([p.frac_x for p in parts]),
                             atomic_numbers=np.concatenate([p.atomic_numbers for p in parts]),
                             lattice=np.concatenate([p.lattice for p in parts]), num_atoms=na,
                             idx_start=np.concatenate([[0], np.cumsum(na)[:-1]]).astype(np.int64))
    else:
        local = SampleResult(frac_x=np.zeros((0, 3)), atomic_numbers=np.zeros(0, dtype=np.int64), lattice=np.zeros((0, 3, 3)),
                             num_atoms=np.zeros(0, dtype=np.int64), idx_start=np.zeros(0, dtype=np.int64))
    t0 = time.perf_counter()
    result = gather_sample_results(local, group=group, device=torch.device(device) if world > 1 else None)
    t1 = time.perf_counter()
    if out_path and rank == 0:
        save_sample_results_to_hdf5(result, out_path)
    if timings is not None:
        timings.update(sample=t_batches, gather=t1 - t0, write=time.perf_counter() - t1)
    return result


def draw_num_atoms(dataset_counts, num_crystals: int, seed: int = 0) -> np.ndarray:
    """Atom counts of `num_crystals` crystals drawn with replacement from the counts of a data set's crystals (its
    empirical distribution, as CDVAE samples them), seeded by `seed`.  The whole set is drawn before it is sharded, so
    it does not depend on the number of ranks."""
    counts = np.asarray(dataset_counts, dtype=np.int64).reshape(-1)
    if counts.size == 0:
        raise ValueError("the data set has no crystals to draw atom counts from")
    return np.random.default_rng(seed).choice(counts, size=num_crystals)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--model_path", type=str, required=True)
    ap.add_argument("--num_crystals", type=int, default=100)
    ap.add_argument("--num_atoms", type=int, default=None, help="atoms per crystal (default 4)")
    ap.add_argument("--num_atoms_from", nargs="+", default=None, metavar="DATA",
                    help="draw every crystal's atom count from these dataset files' counts (.h5 or .npz)")
    ap.add_argument("--seed", type=int, default=0, help="seed of the sampling noise and of the --num_atoms_from draw")
    ap.add_argument("--keyed_noise", action="store_true",
                    help="key every crystal's noise by (seed, its index in the run): the output then does not depend on "
                         "--batch or the number of GPUs")
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--precision", default="fp16", choices=["fp32", "fp16"])
    ap.add_argument("--symbols", nargs="*", default=None, help="constant atomic symbols (use_constant_atomic_symbols)")
    ap.add_argument("--out", default=f"{OUT_DIR}/crystals.h5")
    ap.add_argument("--ori_grid", default=None, help=".npy [16,3] (or .npz with key ori_grid): the orientation grid the "
                    "model was trained with; a reference checkpoint does not carry it (quirk B2)")
    ap.add_argument("--no_strict", action="store_true", help="tolerate model tensors missing from the checkpoint")
    args = ap.parse_args(argv)
    counts = None
    if args.num_atoms_from is not None:
        if args.num_atoms is not None:
            ap.error("--num_atoms_from cannot be combined with --num_atoms")
        if args.symbols is not None:
            ap.error("--num_atoms_from cannot be combined with --symbols (constant symbols fix the atom count)")
        from .diffusion.lattice_dataset import CrystalDataset
        counts = draw_num_atoms(CrystalDataset(args.num_atoms_from).atom_counts(), args.num_crystals, args.seed)
    elif args.num_atoms is None:
        args.num_atoms = 4
    from .lightning_wrappers.diffusion import PONITA_DIFFUSION
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        dist.init_process_group("nccl", device_id=dev)
    grid = None
    if args.ori_grid:
        g = np.load(args.ori_grid)
        grid = g["ori_grid"] if hasattr(g, "files") else g
    model = PONITA_DIFFUSION.load_from_checkpoint(args.model_path, ori_grid=grid, strict=not args.no_strict,
                                                  precision=args.precision)
    res = generate_n_crystals(model, args.num_crystals, args.num_atoms, args.symbols, args.batch, device=dev,
                              seed=args.seed, out_path=args.out, num_atoms=counts, keyed_noise=args.keyed_noise)
    if not dist.is_initialized() or dist.get_rank() == 0:
        print(f"wrote {res.num_atoms.shape[0]} crystals ({res.frac_x.shape[0]} atoms)")
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
