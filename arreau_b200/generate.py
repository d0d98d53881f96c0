"""Mirror of main_diffusion_generate.py:52-94 (generate_n_crystals) on the GPU(s).

    python -m arreau_b200.generate --model_path model.ckpt --num_crystals 1024 --num_atoms 40 [--batch 1024]
    python -m arreau_b200.generate --model_path model.ckpt --num_crystals 1024 --num_atoms_from data/train.h5
    python -m arreau_b200.generate ... --keyed_noise      # the same crystals whatever --batch and the number of GPUs
    python -m arreau_b200.generate ... --elements Li Fe P O     # only these elements (with --num_atoms[_from])
    python -m arreau_b200.generate ... --compositions_from data/test.h5   # structures for the data's compositions
    python -m arreau_b200.generate ... --structures_from data/test.h5 --fix_lattice       # positions in the data's cells
    python -m arreau_b200.generate ... --structures_from data/test.h5 --fix_lattice --free_elements Li   # where Li goes
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
                        keyed_noise: bool = False, elements=None, compositions=None, lattices=None,
                        sites=None) -> SampleResult:
    """main_diffusion_generate.py:52-94.  With torch.distributed initialised the crystals are sharded over the ranks;
    every rank returns the full gathered result and rank 0 writes `out_path`.  `timings` (optional dict) receives this
    rank's wall-clock seconds per phase: `sample` (list, one per batch), `gather`, `write`.  `num_atoms` (optional,
    length num_crystals) gives every crystal its own atom count instead of `num_atoms_per_sample`; each rank samples
    its shard of it (see `draw_num_atoms`).  `keyed_noise`: crystal i of the run gets id i and every draw of its
    trajectory is keyed by (seed, i) on the device (DiffusionLoss.sample's crystal_ids), so the result does not depend
    on num_crystals_per_batch or on the number of ranks.  Without it, batch b0.. is sampled with seed + b0.
    `elements`: one chemical system (element symbols) for every crystal, or a list of num_crystals systems, sharded
    like `num_atoms`; every atom of a crystal ends on an element of its system (PONITA_DIFFUSION.sample's `elements`).
    `compositions`: num_crystals arrays of atomic numbers; each fixes its crystal's atom count and types (crystal
    structure prediction), so it excludes num_atoms, use_constant_atomic_symbols and elements.
    `lattices` (num_crystals 3x3 lattices or None) and `sites` (num_crystals (atomic_numbers, frac) pairs or None) fix
    part of each crystal's structure (PONITA_DIFFUSION.sample's `lattices` / `sites`), sharded like `compositions`."""
    if compositions is not None:
        if num_atoms is not None or use_constant_atomic_symbols is not None or elements is not None:
            raise ValueError("compositions fix atom counts and types: they cannot be combined with num_atoms, "
                             "use_constant_atomic_symbols or elements")
        compositions = [np.asarray(c, dtype=np.int64).reshape(-1) for c in compositions]
        if len(compositions) != num_crystals:
            raise ValueError(f"compositions must hold {num_crystals} crystals, got {len(compositions)}")
        num_atoms = np.asarray([c.size for c in compositions], dtype=np.int64)
    elif num_atoms is not None:
        num_atoms = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
        if num_atoms.shape[0] != num_crystals or np.any(num_atoms < 1):
            raise ValueError(f"num_atoms must hold {num_crystals} positive counts, got {num_atoms.shape[0]}")
        if use_constant_atomic_symbols is not None:
            raise ValueError("constant atomic symbols fix the atom count: they cannot be combined with num_atoms")
    per_crystal_elements = elements is not None and not all(isinstance(e, str) for e in elements)
    if elements is not None:
        if use_constant_atomic_symbols is not None:
            raise ValueError("constant atomic symbols fix the types: they cannot be combined with elements")
        if per_crystal_elements and len(elements) != num_crystals:
            raise ValueError(f"elements must hold one system or {num_crystals} systems, got {len(elements)}")
    for name, per_crystal in (("lattices", lattices), ("sites", sites)):
        if per_crystal is not None and len(per_crystal) != num_crystals:
            raise ValueError(f"{name} must hold {num_crystals} crystals, got {len(per_crystal)}")
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    lo, hi = shard_range(num_crystals, rank, world)
    parts = []
    t_batches = []
    for b0 in range(lo, hi, num_crystals_per_batch):
        nb = min(num_crystals_per_batch, hi - b0)
        if compositions is not None:
            kw = {"compositions": compositions[b0:b0 + nb]}
        else:
            kw = {} if num_atoms is None else {"num_atoms": torch.from_numpy(num_atoms[b0:b0 + nb].copy())}
        if elements is not None:
            kw["elements"] = elements[b0:b0 + nb] if per_crystal_elements else elements
        if lattices is not None:
            kw["lattices"] = lattices[b0:b0 + nb]
        if sites is not None:
            kw["sites"] = sites[b0:b0 + nb]
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


def draw_compositions(dataset, num_crystals: int, seed: int = 0):
    """(indices, compositions) of `num_crystals` crystals of a CrystalDataset drawn with replacement, seeded by `seed`:
    their dataset indices (int64) and their atomic-number arrays.  Drawn before sharding, like draw_num_atoms, so it
    does not depend on the number of ranks; the indices lead back to each composition's ground-truth structure."""
    if len(dataset) == 0:
        raise ValueError("the data set has no crystals to draw compositions from")
    idx = np.random.default_rng(seed).choice(len(dataset), size=num_crystals).astype(np.int64)
    return idx, [np.asarray(dataset.configs[i].atomic_numbers, dtype=np.int64).reshape(-1) for i in idx]


def known_structures(dataset, index, fix_lattice: bool, free_elements=None):
    """(compositions, lattices, sites) of the CrystalDataset crystals `index` for structure-conditioned generation.
    `fix_lattice`: each crystal keeps its lattice (else None).  `free_elements` (element symbols): every atom of
    another element keeps its dataset position as a site, and the composition lists the sites first, then the free
    atoms, in dataset order; None leaves every position free (sites None).  ValueError names an unknown symbol."""
    from .tools.atomic_number_table import ATOMIC_NUMBER
    free_z = None
    if free_elements is not None:
        unknown = [e for e in free_elements if e not in ATOMIC_NUMBER]
        if unknown:
            raise ValueError(f"unknown element symbols {unknown}")
        free_z = [ATOMIC_NUMBER[e] for e in free_elements]
    compositions, lattices, sites = [], [], []
    for i in index:
        cfg = dataset.configs[int(i)]
        z = np.asarray(cfg.atomic_numbers, dtype=np.int64).reshape(-1)
        lattices.append(np.asarray(cfg.L0, dtype=np.float64).reshape(3, 3) if fix_lattice else None)
        if free_z is None:
            compositions.append(z)
            continue
        free = np.isin(z, free_z)
        compositions.append(np.concatenate([z[~free], z[free]]))
        x = np.asarray(cfg.X0, dtype=np.float64).reshape(-1, 3)
        sites.append((z[~free], x[~free]) if (~free).any() else None)
    return compositions, (lattices if fix_lattice else None), (sites if free_z is not None else None)


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
    ap.add_argument("--elements", nargs="+", default=None, metavar="SYMBOL",
                    help="chemical system: every atom of every crystal is one of these elements")
    ap.add_argument("--compositions_from", nargs="+", default=None, metavar="DATA",
                    help="sample structures for compositions drawn (seeded by --seed) from these dataset files' crystals; "
                         "the output file also holds their dataset indices as source_index")
    ap.add_argument("--structures_from", nargs="+", default=None, metavar="DATA",
                    help="sample structures conditioned on crystals drawn (seeded by --seed) from these dataset files: "
                         "their compositions, and with --fix_lattice / --free_elements part of their structure; the "
                         "output file also holds their dataset indices as source_index")
    ap.add_argument("--fix_lattice", action="store_true",
                    help="with --structures_from: every crystal keeps its dataset lattice (structure prediction in a "
                         "known cell)")
    ap.add_argument("--free_elements", nargs="+", default=None, metavar="SYMBOL",
                    help="with --structures_from: the atoms of these elements are generated, every other atom keeps its "
                         "dataset position (structure completion)")
    ap.add_argument("--out", default=f"{OUT_DIR}/crystals.h5")
    ap.add_argument("--ori_grid", default=None, help=".npy [16,3] (or .npz with key ori_grid): the orientation grid the "
                    "model was trained with; a reference checkpoint does not carry it (quirk B2)")
    ap.add_argument("--no_strict", action="store_true", help="tolerate model tensors missing from the checkpoint")
    args = ap.parse_args(argv)
    counts = compositions = source_index = lattices = sites = None
    if args.structures_from is None and (args.fix_lattice or args.free_elements is not None):
        ap.error("--fix_lattice and --free_elements need --structures_from")
    if args.structures_from is not None:
        for opt in ("num_atoms", "num_atoms_from", "symbols", "elements", "compositions_from"):
            if getattr(args, opt) is not None:
                ap.error(f"--structures_from cannot be combined with --{opt} (the structures fix counts and types)")
        if not args.fix_lattice and args.free_elements is None:
            ap.error("--structures_from needs --fix_lattice, --free_elements or both (what to keep of each structure)")
        from .diffusion.lattice_dataset import CrystalDataset
        data = CrystalDataset(args.structures_from)
        source_index, _ = draw_compositions(data, args.num_crystals, args.seed)
        try:
            compositions, lattices, sites = known_structures(data, source_index, args.fix_lattice, args.free_elements)
        except ValueError as e:
            ap.error(str(e))
    elif args.compositions_from is not None:
        for opt in ("num_atoms", "num_atoms_from", "symbols", "elements"):
            if getattr(args, opt) is not None:
                ap.error(f"--compositions_from cannot be combined with --{opt} (the compositions fix counts and types)")
        from .diffusion.lattice_dataset import CrystalDataset
        source_index, compositions = draw_compositions(CrystalDataset(args.compositions_from), args.num_crystals,
                                                       args.seed)
    elif args.elements is not None and args.symbols is not None:
        ap.error("--elements cannot be combined with --symbols (constant symbols fix the types)")
    elif args.num_atoms_from is not None:
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
                              seed=args.seed, num_atoms=counts, keyed_noise=args.keyed_noise, elements=args.elements,
                              compositions=compositions, lattices=lattices, sites=sites)
    if not dist.is_initialized() or dist.get_rank() == 0:
        extra = {} if source_index is None else {"source_index": source_index}
        path = save_sample_results_to_hdf5(res, args.out, extra)
        print(f"wrote {res.num_atoms.shape[0]} crystals ({res.frac_x.shape[0]} atoms) to {path}")
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
