"""Mirror of diffusion/lattice_dataset.py (SURVEY 8f-4): the training input pipeline.

Reads the reference's dataset files -- HDF5 with groups `atomic_number/<i>`, `frac_coord/<i>` and the dataset
`lattice_matrix[G,3,3]` (prep_datasets.py:67-79, lattice_dataset.py:23-42) through h5py when it is installed, or the
same three keys from a NumPy `.npz` (`atomic_number_<i>`, `frac_coord_<i>`, `lattice_matrix`; `save_dataset_npz`
writes it) -- and collates variable-size crystals into the flat batch DiffusionLoss.__call__ consumes:
`Batch{X0[N,3], A0[N], L0[3G,3], num_atoms[G], batch[N]}` (what PyG's DataLoader builds from lattice_dataset.py:98-113).
Collation is host-side index arithmetic on pinned memory followed by ONE asynchronous copy per field, so a training
loop is not bound by per-crystal Python work on the device."""
from __future__ import annotations

import argparse
import os
from dataclasses import dataclass
from typing import List, Sequence

import numpy as np
import torch

from ..tools.atomic_number_table import AtomicNumberTable


@dataclass
class Configuration:
    """lattice_dataset.py:15-20."""
    atomic_numbers: np.ndarray
    X0: np.ndarray
    L0: np.ndarray


def load_data(filename: str):
    """lattice_dataset.py:23-42 (HDF5), or the .npz twin."""
    if filename.endswith(".npz"):
        z = np.load(filename)
        lattice = np.asarray(z["lattice_matrix"])
        n = lattice.shape[0]
        return [np.asarray(z[f"atomic_number_{i}"]) for i in range(n)], lattice, [np.asarray(z[f"frac_coord_{i}"]) for i in range(n)]
    import h5py   # the reference's format; not part of this image
    with h5py.File(filename, "r") as f:
        keys = sorted(f["atomic_number"], key=int)
        zs = [np.array(f["atomic_number"][k]) for k in keys]
        lattice = np.array(f["lattice_matrix"])
        keys = sorted(f["frac_coord"], key=int)
        frac = [np.array(f["frac_coord"][k]) for k in keys]
    return zs, lattice, frac


def save_dataset_npz(filename: str, atomic_number_vectors, lattice_matrices, frac_coords_arrays) -> str:
    """prep_datasets.py:67-79 for environments without h5py."""
    path = filename if filename.endswith(".npz") else filename + ".npz"
    os.makedirs(os.path.dirname(os.path.abspath(path)) or ".", exist_ok=True)
    arrays = {"lattice_matrix": np.asarray(lattice_matrices)}
    for i, (z, x) in enumerate(zip(atomic_number_vectors, frac_coords_arrays)):
        arrays[f"atomic_number_{i}"] = np.asarray(z)
        arrays[f"frac_coord_{i}"] = np.asarray(x)
    np.savez(path, **arrays)
    return path


def load_dataset(file_path: str) -> List[Configuration]:
    """lattice_dataset.py:45-58."""
    zs, lattice, frac = load_data(file_path)
    out = []
    for i in range(len(lattice)):
        assert lattice[i].shape == (3, 3)
        out.append(Configuration(atomic_numbers=zs[i], X0=frac[i], L0=lattice[i]))
    return out


class CrystalDataset(torch.utils.data.Dataset):
    """lattice_dataset.py:75-113: all configurations in memory, the z_table from the atomic numbers that occur
    (+ the mask state 2001)."""

    def __init__(self, config_paths: Sequence[str], cutoff: float = 5.0):
        self.configs = [c for p in config_paths for c in load_dataset(p)]
        zs = set()
        for c in self.configs:
            zs.update(int(z) for z in np.asarray(c.atomic_numbers).reshape(-1))
        zs.add(AtomicNumberTable.MASK_ATOMIC_NUMBER)
        self.unique_atomic_numbers = zs
        self.z_table = AtomicNumberTable(sorted(zs))
        self.cutoff = cutoff
        self._index = {z: i for i, z in enumerate(self.z_table.zs)}
        # flat copy of the whole set for the epoch iterator (`collate_indices`): one gather per field instead of a Python
        # loop over the atoms of every crystal of every batch
        na = np.asarray([len(np.asarray(c.atomic_numbers).reshape(-1)) for c in self.configs], dtype=np.int64)
        self._na = na
        self._off = np.concatenate([[0], np.cumsum(na)]).astype(np.int64)
        if len(self.configs):
            lut = np.full(max(zs) + 1, -1, dtype=np.int64)
            for z, i in self._index.items():
                lut[z] = i
            self._A0 = lut[np.concatenate([np.asarray(c.atomic_numbers).reshape(-1).astype(np.int64) for c in self.configs])]
            self._X0 = np.concatenate([np.asarray(c.X0, dtype=np.float64).reshape(-1, 3) for c in self.configs])
            self._L0 = np.stack([np.asarray(c.L0, dtype=np.float64) for c in self.configs])

    def collate_indices(self, indices, device=None, pin: bool = True):
        """`collate_crystals([self[i] for i in indices])` as vectorised gathers over the flat copy (same fields, same values)."""
        b = np.asarray(indices, dtype=np.int64).reshape(-1)
        na = self._na[b]
        total = int(na.sum())
        # positions of the selected crystals' atoms in the flat arrays: start of each crystal repeated, plus a running index
        starts = self._off[b]
        within = np.arange(total, dtype=np.int64) - np.repeat(np.cumsum(na) - na, na)
        idx = np.repeat(starts, na) + within
        X0, A0 = self._X0[idx], self._A0[idx]
        L0m = self._L0[b]
        batch = np.repeat(np.arange(len(b)), na)
        pos = np.einsum("bi,bij->bj", X0, L0m[batch])
        return _to_namespace(dict(X0=X0, A0=A0, L0=L0m.reshape(-1, 3), num_atoms=na, batch=batch, pos=pos), device, pin)

    def atom_counts(self) -> np.ndarray:
        """Atoms per crystal, in dataset order."""
        return self._na

    def __len__(self):
        return len(self.configs)

    def __getitem__(self, idx: int):
        c = self.configs[idx]
        A0 = np.asarray([self._index[int(z)] for z in np.asarray(c.atomic_numbers).reshape(-1)], dtype=np.int64)
        return dict(X0=np.asarray(c.X0, dtype=np.float64), A0=A0, L0=np.asarray(c.L0, dtype=np.float64), num_atoms=len(A0))


class CrystalSubset(torch.utils.data.Dataset):
    """The crystals `indices` of a CrystalDataset (a train / valid / test split) with the parent's z_table and collation.
    `crystal_ids` are the crystals' indices in the parent: the evaluation noise is keyed by them, so a crystal draws the
    same numbers whichever split view, batch or rank it is evaluated in."""

    def __init__(self, parent: CrystalDataset, indices):
        self.parent = parent
        self.crystal_ids = np.asarray(indices, dtype=np.int64).reshape(-1)
        self.z_table = parent.z_table

    def collate_indices(self, indices, device=None, pin: bool = True):
        return self.parent.collate_indices(self.crystal_ids[np.asarray(indices, dtype=np.int64)], device=device, pin=pin)

    def atom_counts(self) -> np.ndarray:
        return self.parent.atom_counts()[self.crystal_ids]

    def __len__(self):
        return int(self.crystal_ids.shape[0])

    def __getitem__(self, idx: int):
        return self.parent[int(self.crystal_ids[idx])]


def split_indices(n: int, fractions: Sequence[float], seed: int = 0) -> List[np.ndarray]:
    """Seeded split of range(n) into len(fractions) disjoint parts that together cover it (fractions sum to 1): part k
    takes the next round(n * (f_0 + .. + f_k)) - round(n * (f_0 + .. + f_{k-1})) entries of one seeded permutation.
    Each part is returned in ascending order."""
    f = np.asarray(fractions, dtype=np.float64).reshape(-1)
    if f.size == 0 or np.any(f < 0) or abs(float(f.sum()) - 1.0) > 1e-9:
        raise ValueError(f"fractions must be non-negative and sum to 1, got {list(f)}")
    bounds = np.round(n * np.cumsum(f)).astype(np.int64)
    bounds[-1] = n
    order = np.random.default_rng(seed).permutation(n)
    return [np.sort(p) for p in np.split(order, bounds[:-1])]


def collate_crystals(items: Sequence[dict], device=None, pin: bool = True):
    """PyG-style collation of `CrystalDataset` items into the flat batch of DiffusionLoss.__call__
    (diffusion_loss.py:205-209): X0[N,3], A0[N], L0[3G,3], num_atoms[G], batch[N], pos[N,3] = X0 @ L0."""
    na = np.asarray([it["num_atoms"] for it in items], dtype=np.int64)
    X0 = np.concatenate([it["X0"] for it in items]).astype(np.float64)
    A0 = np.concatenate([it["A0"] for it in items]).astype(np.int64)
    L0 = np.concatenate([it["L0"] for it in items]).astype(np.float64)              # [3G,3] like PyG's cat of [3,3]
    batch = np.repeat(np.arange(len(items)), na)
    pos = np.einsum("bi,bij->bj", X0, L0.reshape(-1, 3, 3)[batch])
    return _to_namespace(dict(X0=X0, A0=A0, L0=L0, num_atoms=na, batch=batch, pos=pos), device, pin)


def _to_namespace(fields: dict, device, pin: bool):
    out = {}
    for k, v in fields.items():
        t = torch.from_numpy(np.ascontiguousarray(v))
        if device is not None and torch.device(device).type == "cuda":
            t = (t.pin_memory() if pin else t).to(device, non_blocking=True)
        out[k] = t
    # the atoms-per-crystal vector stays available on the host: the engines bind the batch topology from it without a
    # device -> host read (which would synchronise every training step)
    out["num_atoms_cpu"] = np.asarray(fields["num_atoms"], dtype=np.int64).copy()
    return argparse.Namespace(**out)


def batches(dataset: CrystalDataset, batch_size: int, shuffle: bool = True, seed: int = 0, device=None, rank: int = 0,
            world: int = 1):
    """Epoch iterator: shuffles, shards the batches over `world` ranks (DDP's DistributedSampler role) and collates.
    Every rank gets the SAME number of batches -- each training step carries a gradient all-reduce, so a rank that ran
    out of batches early would leave its peers in a collective it never joins: like torch's DistributedSampler
    (drop_last=False) the list of batches is padded to a multiple of `world` by wrapping around to the first ones."""
    for b in batch_index_lists(len(dataset), batch_size, shuffle, seed, rank, world):
        if hasattr(dataset, "collate_indices"):
            yield dataset.collate_indices(b, device=device)
        else:
            yield collate_crystals([dataset[int(i)] for i in b], device=device)


def batch_index_lists(n: int, batch_size: int, shuffle: bool = True, seed: int = 0, rank: int = 0, world: int = 1):
    """Dataset indices of this rank's batches for one epoch (see `batches`); identical length on every rank."""
    if n == 0:
        return []
    order = np.random.default_rng(seed).permutation(n) if shuffle else np.arange(n)
    all_batches = [order[s:s + batch_size] for s in range(0, n, batch_size)]
    pad = (-len(all_batches)) % world
    all_batches += [all_batches[i % len(all_batches)] for i in range(pad)]
    return all_batches[rank::world]
