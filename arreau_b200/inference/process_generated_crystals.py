"""Mirror of diffusion/inference/process_generated_crystals.py:8-33: the wire format of generated crystals.

Layout (group "crystals"): frac_x[N,3] f64, atomic_numbers[N], lattice[G,3,3] f64, idx_start[G], num_atoms[G].
HDF5 through h5py when it is installed (the reference's format, byte-compatible readers); otherwise -- h5py is not
part of this image -- the same five arrays under the same keys ("crystals/<name>") in a NumPy .npz archive."""
from __future__ import annotations

import os
from typing import Optional

import numpy as np

from ..diffusion.diffusion_loss import SampleResult

KEYS = ("frac_x", "atomic_numbers", "lattice", "idx_start", "num_atoms")


def _have_h5py() -> bool:
    try:
        import h5py  # noqa: F401
        return True
    except Exception:
        return False


def save_sample_results_to_hdf5(crystals: SampleResult, filename: str, extra: Optional[dict] = None) -> str:
    """process_generated_crystals.py:8-15.  Returns the path actually written (".npz" replaces ".h5" without h5py).
    `extra`: further arrays stored next to the five (e.g. `source_index` of generate --compositions_from); readers
    that take the five keys are unaffected."""
    os.makedirs(os.path.dirname(os.path.abspath(filename)) or ".", exist_ok=True)
    arrays = {**{k: getattr(crystals, k) for k in KEYS}, **(extra or {})}
    if _have_h5py() and not filename.endswith(".npz"):
        import h5py
        with h5py.File(filename, "w") as file:
            group = file.create_group("crystals")
            for k, v in arrays.items():
                group.create_dataset(k, data=v)
        return filename
    path = filename if filename.endswith(".npz") else os.path.splitext(filename)[0] + ".npz"
    np.savez(path, **{f"crystals/{k}": np.asarray(v) for k, v in arrays.items()})
    return path


def load_sample_results_from_hdf5(filename: str) -> SampleResult:
    """process_generated_crystals.py:18-31 (path taken as given)."""
    if filename.endswith(".npz") or not _have_h5py():
        path = filename if filename.endswith(".npz") else os.path.splitext(filename)[0] + ".npz"
        z = np.load(path)
        return SampleResult(**{k: z[f"crystals/{k}"] for k in KEYS})
    import h5py
    with h5py.File(filename, "r") as file:
        return SampleResult(**{k: file["crystals"][k][:] for k in KEYS})


def load_extra_arrays(filename: str, keys) -> dict:
    """The arrays among `keys` stored next to the five by save_sample_results_to_hdf5(extra=...) (e.g. source_index),
    by key; a key the file lacks is left out."""
    if filename.endswith(".npz") or not _have_h5py():
        path = filename if filename.endswith(".npz") else os.path.splitext(filename)[0] + ".npz"
        z = np.load(path)
        return {k: z[f"crystals/{k}"] for k in keys if f"crystals/{k}" in z.files}
    import h5py
    with h5py.File(filename, "r") as file:
        return {k: file["crystals"][k][:] for k in keys if k in file["crystals"]}


def get_crystal_indexes(sample_result: SampleResult, sample_idx: int):
    """process_generated_crystals.py:34-38."""
    start = sample_result.idx_start[sample_idx]
    return start, start + sample_result.num_atoms[sample_idx]
