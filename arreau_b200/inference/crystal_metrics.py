"""Quality metrics of generated crystals on the GPU: CDVAE / DiffCSP structural validity and property statistics.

    python -m arreau_b200.inference.crystal_metrics out/crystals.h5 --reference data/test.h5 [--json metrics.json]

Per crystal (`crystal_metrics`, one `arreau_crystal_metrics` launch per chunk): the cell volume, the exact
minimum-image distance over distinct atom pairs, the density and the number of distinct elements, with flags.  A
crystal is structurally valid when every pair of distinct atoms is at least 0.5 A apart under periodic boundary
conditions and the cell volume is at least 0.1 A^3 (CDVAE's `structure_validity`).  `summarize` turns the per-crystal
values into the valid fractions and the Wasserstein-1 distances of density, element count and atom count against a
reference set (the data the model was trained on, or its test split).  `quality_record` is the compact subset that
train.fit's sample-quality monitoring logs per pass (the per-crystal rows of all ranks are gathered with
distributed.gather_crystal_metrics first).  `system_fractions` checks generated crystals against a chemical system
(generate --elements) on the host.  With --match the crystals are also matched against their source structures
(structure_match.py: CSP match rate and RMSE).  With --unique_novel they are grouped by pymatgen's
StructureMatcher.fit (group_structures: uniqueness) and matched against the --reference crystals of the same
composition (novelty), on the GPU matcher (structure_match.py).  Compositional validity (oxidation states) and
coverage need SMACT / CrystalNN and are not computed here."""
from __future__ import annotations

import argparse
import json
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from .. import _lib
from ..diffusion.diffusion_loss import SampleResult
from ..tools.atomic_number_table import ATOMIC_MASS, ATOMIC_NUMBER
from .process_generated_crystals import load_sample_results_from_hdf5

# bits of CrystalMetrics.flags (ARREAU_METRICS_* in include/arreau_b200.h)
VALID, UNKNOWN_ELEMENT, DEGENERATE, EXTENDED_SEARCH = 1, 2, 4, 8
# atoms per launch: bounds the device memory of a chunk (~24 bytes per atom of input) for data sets of any size
MAX_CHUNK_ATOMS = 1 << 22


@dataclass
class CrystalMetrics:
    """Per-crystal metrics, numpy arrays of length G.  min_dist is +inf below two atoms and NaN for a degenerate cell;
    density is NaN when an element is unknown (Z outside 1..103, e.g. the D3PM mask state 2001)."""
    num_atoms: np.ndarray      # int64
    volume: np.ndarray         # A^3
    min_dist: np.ndarray       # A
    density: np.ndarray        # g/cm^3
    num_elements: np.ndarray   # int32, distinct known Z
    flags: np.ndarray          # int32, VALID | UNKNOWN_ELEMENT | DEGENERATE | EXTENDED_SEARCH

    @property
    def valid(self) -> np.ndarray:
        return (self.flags & VALID) != 0

    @property
    def known(self) -> np.ndarray:
        return (self.flags & UNKNOWN_ELEMENT) == 0

    @property
    def degenerate(self) -> np.ndarray:
        return (self.flags & DEGENERATE) != 0

    @property
    def extended_search(self) -> np.ndarray:
        return (self.flags & EXTENDED_SEARCH) != 0


_MASS_TABLES = {}
_NUMPY_DTYPE = {torch.float64: np.float64, torch.int64: np.int64, torch.int32: np.int32}


def _mass_table(dev: torch.device) -> torch.Tensor:
    """ATOMIC_MASS indexed by Z (entry 0 = unknown) on `dev`, uploaded once per device."""
    key = str(dev)
    if key not in _MASS_TABLES:
        _MASS_TABLES[key] = torch.tensor((0.0,) + tuple(ATOMIC_MASS), dtype=torch.float64).to(dev)
    return _MASS_TABLES[key]


def _rows_on(x, lo: int, hi: int, dtype: torch.dtype, dev: torch.device) -> torch.Tensor:
    """Rows lo:hi of a numpy array or tensor as a contiguous `dtype` tensor on `dev`: a tensor already there is used
    as it is, host data goes through pinned memory."""
    if isinstance(x, torch.Tensor):
        t = x[lo:hi]
        if t.device != dev:
            t = (t.pin_memory() if t.device.type == "cpu" else t).to(dev, non_blocking=True)
        return t.to(dtype).contiguous()
    a = np.ascontiguousarray(np.asarray(x)[lo:hi], dtype=_NUMPY_DTYPE[dtype])
    return torch.from_numpy(a).pin_memory().to(dev, non_blocking=True)


def _cuda_device(device, what: str) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError(f"{what} runs on a CUDA device")
    return torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev


def _check_inputs(frac_x, lattice, atomic_numbers, num_atoms):
    """num_atoms as int64 and the atom offsets (G + 1 prefix sums), after checking the shapes of the four arrays."""
    na = np.asarray(num_atoms.cpu() if isinstance(num_atoms, torch.Tensor) else num_atoms, dtype=np.int64).reshape(-1)
    G, N = int(na.shape[0]), int(na.sum())
    if np.any(na < 0):
        raise ValueError("num_atoms must be non-negative")
    if tuple(frac_x.shape) != (N, 3) or tuple(lattice.shape) != (G, 3, 3) or tuple(atomic_numbers.shape) != (N,):
        raise ValueError(f"expected frac_x[{N},3], lattice[{G},3,3], atomic_numbers[{N}]; got {tuple(frac_x.shape)}, "
                         f"{tuple(lattice.shape)}, {tuple(atomic_numbers.shape)}")
    if N >= 2 ** 31:
        raise ValueError("at most 2^31 - 1 atoms")
    off = np.zeros(G + 1, dtype=np.int64)
    np.cumsum(na, out=off[1:])
    return na, off


def _run_chunked(off, max_chunk_atoms: int, dtypes, launch, dev: torch.device):
    """Per-crystal outputs of a kernel run over chunks of crystals of at most `max_chunk_atoms` atoms by the prefix
    sums `off` (a larger crystal is a chunk of its own).  launch(g0, g1, ptrs, stream) enqueues crystals g0:g1 with
    one output pointer per entry of `dtypes`; the outputs of a chunk share one device buffer and one device->host
    read.  Returns one host array per dtype."""
    G = len(off) - 1
    items = [np.dtype(dt).itemsize for dt in dtypes]
    ends = np.cumsum([0] + items)
    views = [np.empty(G, dtype=dt) for dt in dtypes]
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        g0 = 0
        while g0 < G:
            g1 = int(np.searchsorted(off, off[g0] + max_chunk_atoms, side="right")) - 1
            g1 = min(max(g1, g0 + 1), G)
            Gc = g1 - g0
            out = torch.empty(Gc * int(ends[-1]), dtype=torch.uint8, device=dev)
            launch(g0, g1, [out[Gc * int(lo):].data_ptr() for lo in ends[:-1]], stream)
            chunk = out.cpu().numpy()
            for v, lo, hi, dt in zip(views, ends[:-1], ends[1:], dtypes):
                v[g0:g1] = chunk[Gc * lo:Gc * hi].view(dt)
            g0 = g1
    return views


def crystal_metrics(frac_x, lattice, atomic_numbers, num_atoms, device="cuda", min_dist: float = 0.5,
                    min_volume: float = 0.1, max_chunk_atoms: int = MAX_CHUNK_ATOMS) -> CrystalMetrics:
    """Metrics of G crystals stored back to back: frac_x[N,3], lattice[G,3,3] (rows a, b, c; pos = frac @ lattice),
    atomic_numbers[N] (Z), num_atoms[G].  Each may be a numpy array or a tensor; tensors on `device` are read in
    place.  The crystals are processed in chunks of at most `max_chunk_atoms` atoms (a larger crystal is a chunk of
    its own), each with one device->host read; a crystal's results do not depend on the chunking.  `min_dist` (A) and
    `min_volume` (A^3) are the validity thresholds."""
    dev = _cuda_device(device, "crystal_metrics")
    na, off = _check_inputs(frac_x, lattice, atomic_numbers, num_atoms)

    def launch(g0, g1, outs, stream):
        a0, a1, Gc = int(off[g0]), int(off[g1]), g1 - g0
        f = _rows_on(frac_x, a0, a1, torch.float64, dev)
        lat = _rows_on(lattice, g0, g1, torch.float64, dev)
        z = _rows_on(atomic_numbers, a0, a1, torch.int64, dev)
        o = _rows_on((off[g0:g1 + 1] - a0).astype(np.int32), 0, Gc + 1, torch.int32, dev)
        mass = _mass_table(dev)
        _lib.call("arreau_crystal_metrics", f.data_ptr(), lat.data_ptr(), z.data_ptr(), o.data_ptr(), a1 - a0, Gc,
                  mass.data_ptr(), mass.shape[0] - 1, float(min_dist), float(min_volume), *outs, stream)

    views = _run_chunked(off, max_chunk_atoms, (np.float64, np.float64, np.float64, np.int32, np.int32), launch, dev)
    return CrystalMetrics(num_atoms=na, volume=views[0], min_dist=views[1], density=views[2], num_elements=views[3],
                          flags=views[4])


def sample_inputs(samples):
    """(frac_x, lattice, atomic_numbers, num_atoms) of a SampleResult, or of a crystals file written by `generate`
    (load_sample_results_from_hdf5)."""
    res: SampleResult = load_sample_results_from_hdf5(samples) if isinstance(samples, str) else samples
    na = np.asarray(res.num_atoms, dtype=np.int64).reshape(-1)
    if res.idx_start is not None:
        start = np.concatenate([[0], np.cumsum(na)[:-1]]).astype(np.int64)
        if not np.array_equal(np.asarray(res.idx_start, dtype=np.int64).reshape(-1), start):
            raise ValueError("crystals must be stored back to back (idx_start = exclusive cumsum of num_atoms)")
    return (np.asarray(res.frac_x, dtype=np.float64).reshape(-1, 3),
            np.asarray(res.lattice, dtype=np.float64).reshape(-1, 3, 3),
            np.asarray(res.atomic_numbers, dtype=np.int64).reshape(-1), na)


def dataset_inputs(dataset):
    """(frac_x, lattice, atomic_numbers, num_atoms) of a CrystalDataset or CrystalSubset, in its order; the atomic
    numbers come from the data set's z_table."""
    if len(dataset) == 0:
        return np.zeros((0, 3)), np.zeros((0, 3, 3)), np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    b = dataset.collate_indices(np.arange(len(dataset)), device=None)
    zs = np.asarray(dataset.z_table.zs, dtype=np.int64)
    return b.X0.numpy(), b.L0.numpy().reshape(-1, 3, 3), zs[b.A0.numpy()], b.num_atoms.numpy()


def _w1(a, b) -> Optional[float]:
    from scipy.stats import wasserstein_distance
    return float(wasserstein_distance(a, b)) if len(a) and len(b) else None


def _frac(k: int, n: int) -> Optional[float]:
    return k / n if n else None


def summarize(generated: CrystalMetrics, reference: Optional[CrystalMetrics] = None) -> dict:
    """Summary of generated crystals (JSON-ready; None where a set is empty):
    - counts and fractions of valid, unknown-element and degenerate crystals, and of those that needed the extended
      image search;
    - percentiles of min_dist over the crystals with a finite one (two or more atoms, not degenerate);
    - mean density and element count over the valid crystals with known elements.
    With a reference (CDVAE's convention): w1_density and w1_num_elements between the valid generated crystals with
    known elements and every reference crystal with known elements, w1_num_atoms between all generated and all
    reference crystals, and the reference's own valid fraction (about 1 for real crystals)."""
    G = int(generated.flags.shape[0])
    valid, known = generated.valid, generated.known
    sel = valid & known
    finite = np.isfinite(generated.min_dist)
    out = dict(num_crystals=G, num_valid=int(valid.sum()), frac_valid=_frac(int(valid.sum()), G),
               num_unknown_element=int((~known).sum()), frac_unknown_element=_frac(int((~known).sum()), G),
               num_degenerate=int(generated.degenerate.sum()), frac_degenerate=_frac(int(generated.degenerate.sum()), G),
               num_extended_search=int(generated.extended_search.sum()))
    for p in (1, 5, 25, 50):
        out[f"min_dist_p{p}"] = float(np.percentile(generated.min_dist[finite], p)) if finite.any() else None
    out["mean_density"] = float(generated.density[sel].mean()) if sel.any() else None
    out["mean_num_elements"] = float(generated.num_elements[sel].mean()) if sel.any() else None
    if reference is not None:
        rk = reference.known
        R = int(reference.flags.shape[0])
        out.update(reference_num_crystals=R, reference_frac_valid=_frac(int(reference.valid.sum()), R),
                   w1_density=_w1(generated.density[sel], reference.density[rk]),
                   w1_num_elements=_w1(generated.num_elements[sel], reference.num_elements[rk]),
                   w1_num_atoms=_w1(generated.num_atoms, reference.num_atoms))
    return out


def system_fractions(atomic_numbers, num_atoms, elements) -> dict:
    """How well crystals stored back to back (atomic_numbers[N], num_atoms[G]) keep to the chemical system `elements`
    (element symbols): frac_in_system, the share of crystals whose every atom is an element of the system, and
    frac_full_system, the share in which every element of the system occurs (None for no crystals).  Host only."""
    unknown = [e for e in elements if e not in ATOMIC_NUMBER]
    if unknown or len(elements) == 0:
        raise ValueError(f"not a chemical system: unknown element symbols {unknown}" if unknown else "empty chemical system")
    system = np.unique([ATOMIC_NUMBER[e] for e in elements])
    z = np.asarray(atomic_numbers, dtype=np.int64).reshape(-1)
    na = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
    if int(na.sum()) != z.shape[0] or np.any(na < 0):
        raise ValueError(f"num_atoms (sum {int(na.sum())}) does not describe {z.shape[0]} atoms")
    G = int(na.shape[0])
    crystal = np.repeat(np.arange(G), na)
    inside = np.isin(z, system)
    outside = np.zeros(G, dtype=np.int64)
    np.add.at(outside, crystal, ~inside)
    present = np.zeros((G, system.size), dtype=np.bool_)
    present[crystal[inside], np.searchsorted(system, z[inside])] = True
    return dict(frac_in_system=_frac(int((outside == 0).sum()), G),
                frac_full_system=_frac(int(present.all(axis=1).sum()), G))


METRIC_FIELDS = ("num_atoms", "volume", "min_dist", "density", "num_elements", "flags")
_FIELD_DTYPES = (np.int64, np.float64, np.float64, np.float64, np.int32, np.int32)
# the compact record of one sample-quality pass of train.fit (its `sample_quality` history): the epoch and these keys
# of `summarize` against the reference split
QUALITY_KEYS = ("frac_valid", "w1_density", "w1_num_elements", "min_dist_p1", "min_dist_p5", "min_dist_p25",
                "min_dist_p50")


def metrics_from_rows(rows) -> CrystalMetrics:
    """CrystalMetrics from its METRIC_FIELDS arrays in that order (e.g. as all_gather_rows returns them, integers
    widened to int64), each cast back to the field's dtype."""
    return CrystalMetrics(**{k: np.asarray(v).astype(dt, copy=False).reshape(-1)
                             for k, v, dt in zip(METRIC_FIELDS, rows, _FIELD_DTYPES)})


def concat_metrics(parts) -> CrystalMetrics:
    """The crystals of several CrystalMetrics, in order (no parts: an empty one)."""
    return metrics_from_rows([np.concatenate([getattr(p, k) for p in parts]) if parts else np.zeros(0)
                              for k in METRIC_FIELDS])


def quality_record(summary: dict, epoch: int) -> dict:
    """{epoch, frac_valid, w1_density, w1_num_elements, min_dist_p1 .. p50} of a `summarize` result (None where it has
    none)."""
    return {"epoch": int(epoch), **{k: summary.get(k) for k in QUALITY_KEYS}}


def main(argv=None):
    ap = argparse.ArgumentParser(description="Structural validity and property statistics of generated crystals")
    ap.add_argument("samples", help="crystals written by arreau_b200.generate (out/crystals.h5 or .npz)")
    ap.add_argument("--reference", nargs="+", default=None, metavar="DATA",
                    help="dataset files (.h5 as written by prep_datasets.py, or .npz) to compare the distributions with")
    ap.add_argument("--json", default=None, metavar="PATH", help="also write the summary as JSON")
    ap.add_argument("--elements", nargs="+", default=None, metavar="SYMBOL",
                    help="chemical system the crystals were generated in: adds frac_in_system and frac_full_system")
    ap.add_argument("--match", action="store_true",
                    help="match every generated crystal against its source structure (the samples' source_index into "
                         "--reference, which must be the files generate drew from): adds match_rate and mean_rms")
    ap.add_argument("--unique_novel", action="store_true",
                    help="group the crystals with pymatgen's StructureMatcher.fit (default tolerances) and match them "
                         "against --reference, normally the training files: adds frac_unique, frac_novel, "
                         "frac_unique_novel and num_new_formula")
    args = ap.parse_args(argv)
    if args.match and not args.reference:
        ap.error("--match needs --reference (the data files generate drew the compositions or structures from)")
    if args.unique_novel and not args.reference:
        ap.error("--unique_novel needs --reference (the data files novelty is measured against, normally the "
                 "training files)")
    from ..diffusion.lattice_dataset import CrystalDataset
    from .process_generated_crystals import load_extra_arrays
    from .structure_match import (check_source_index, match_summary, select_crystals, structure_match, unique_novel,
                                  unique_novel_summary)
    inputs = sample_inputs(args.samples)
    ref_inputs = dataset_inputs(CrystalDataset(args.reference)) if args.reference else None
    source_index = None
    if args.match:
        try:
            source_index = check_source_index(load_extra_arrays(args.samples, ("source_index",)).get("source_index"),
                                              len(inputs[3]), len(ref_inputs[3]))
        except ValueError as e:
            ap.error(str(e))
    generated = crystal_metrics(*inputs)
    reference = crystal_metrics(*ref_inputs) if ref_inputs is not None else None
    summary = summarize(generated, reference)
    if args.elements:
        summary.update(system_fractions(inputs[2], inputs[3], args.elements))
    if args.match:
        summary.update(match_summary(structure_match(inputs, select_crystals(ref_inputs, source_index)), generated))
    if args.unique_novel:
        summary.update(unique_novel_summary(unique_novel(inputs, generated, ref_inputs)))
    for k, v in summary.items():
        print(f"{k}: {v}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(summary, f, indent=1)
    return summary


if __name__ == "__main__":
    main()
