"""Match rate and RMSE of generated crystals against their source structures (crystal structure prediction), on the GPU.

    python -m arreau_b200.inference.crystal_metrics out/crystals.h5 --reference DATA --match

`structure_match` pairs generated crystal i with source crystal i and runs `arreau_structure_match` (csrc/match.cu):
pymatgen's StructureMatcher(stol=0.5, ltol=0.3, angle_tol=10, scale=True, attempt_supercell=False).get_rms_dist as
DiffCSP calls it, without the primitive-cell reduction.  `match_summary` gives DiffCSP's match rate (matched and
structurally valid over all pairs) and the mean RMSE over the matched pairs.  The semantics, the deviations from
pymatgen and the measured speed are in DESIGN.md section 6."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from .. import _lib
from .crystal_metrics import MAX_CHUNK_ATOMS, CrystalMetrics, _check_inputs, _cuda_device, _rows_on, _run_chunked

# bits of StructureMatch.flags (ARREAU_MATCH_* in include/arreau_b200.h)
MATCHED, COMPOSITION, DEGENERATE, SEARCH_LIMIT, TOO_LARGE = 1, 2, 4, 8, 16
MAX_ATOMS = 256


@dataclass
class StructureMatch:
    """Per-pair results, numpy arrays of length G.  rms and max_dist are normalised by (n / V)^(1/3) of the average
    lattice, as pymatgen's; NaN where no candidate was found or the pair was not searched."""
    matched: np.ndarray        # bool, rms < stol
    rms: np.ndarray
    max_dist: np.ndarray
    num_mappings: np.ndarray   # int32, lattice mappings of the generated cell onto the source cell
    flags: np.ndarray          # int32, MATCHED | COMPOSITION | DEGENERATE | SEARCH_LIMIT | TOO_LARGE


def _sorted_by_z(inputs):
    """(frac, lattice, z, num_atoms) on the host with each crystal's atoms stably sorted by Z."""
    frac, lattice, z, na = (np.asarray(a.cpu() if isinstance(a, torch.Tensor) else a) for a in inputs)
    frac = np.asarray(frac, dtype=np.float64).reshape(-1, 3)
    z = np.asarray(z, dtype=np.int64).reshape(-1)
    crystal = np.repeat(np.arange(len(na)), np.asarray(na, dtype=np.int64))
    order = np.lexsort((z, crystal))          # stable: equal Z keep their order
    return frac[order], np.asarray(lattice, dtype=np.float64), z[order], na


def structure_match(gen_inputs, ref_inputs, stol: float = 0.5, ltol: float = 0.3, angle_tol: float = 10.0,
                    device="cuda", max_chunk_atoms: int = MAX_CHUNK_ATOMS) -> StructureMatch:
    """Generated crystal i of `gen_inputs` against crystal i of `ref_inputs`; both are (frac_x[N,3], lattice[G,3,3],
    atomic_numbers[N], num_atoms[G]) as `sample_inputs` / `dataset_inputs` return them, with the same G.  The pairs
    run in chunks of at most `max_chunk_atoms` atoms of both sets together, one device->host read each; a pair's
    results do not depend on the chunking.  stol (in units of (V / n)^(1/3)), ltol (fractional) and angle_tol
    (degrees) are the StructureMatcher tolerances."""
    dev = _cuda_device(device, "structure_match")
    for name, v in (("stol", stol), ("ltol", ltol), ("angle_tol", angle_tol)):
        if not (np.isfinite(v) and v > 0):
            raise ValueError(f"{name} must be finite and positive, got {v}")
    na1, off1 = _check_inputs(*gen_inputs)
    na2, off2 = _check_inputs(*ref_inputs)
    if na1.shape != na2.shape:
        raise ValueError(f"{na1.shape[0]} generated crystals against {na2.shape[0]} source crystals")
    f1, lat1, z1, _ = _sorted_by_z(gen_inputs)
    f2, lat2, z2, _ = _sorted_by_z(ref_inputs)

    def launch(g0, g1, outs, stream):
        a0, a1, b0, b1, Gc = int(off1[g0]), int(off1[g1]), int(off2[g0]), int(off2[g1]), g1 - g0
        args = []
        for f, lat, z, off, lo, hi in ((f1, lat1, z1, off1, a0, a1), (f2, lat2, z2, off2, b0, b1)):
            args.append((_rows_on(f, lo, hi, torch.float64, dev), _rows_on(lat, g0, g1, torch.float64, dev),
                         _rows_on(z, lo, hi, torch.int64, dev),
                         _rows_on((off[g0:g1 + 1] - lo).astype(np.int32), 0, Gc + 1, torch.int32, dev)))
        _lib.call("arreau_structure_match", *[t.data_ptr() for t in args[0]], *[t.data_ptr() for t in args[1]],
                  a1 - a0, b1 - b0, Gc, float(stol), float(ltol), float(angle_tol), *outs, stream)

    rms, max_dist, num_mappings, flags = _run_chunked(off1 + off2, max_chunk_atoms,
                                                      (np.float64, np.float64, np.int32, np.int32), launch, dev)
    return StructureMatch(matched=(flags & MATCHED) != 0, rms=rms, max_dist=max_dist, num_mappings=num_mappings,
                          flags=flags)


def match_summary(match: StructureMatch, generated: CrystalMetrics) -> dict:
    """DiffCSP's CSP summary (JSON-ready; None where a set is empty): match_rate, the share of all pairs whose
    generated crystal matches its source and is structurally valid with known elements (crystal_metrics), mean_rms
    over those pairs, and the counts of pairs with a composition mismatch (a generated atom left in the mask state is
    one), a search limit, a degenerate cell or a crystal above 256 atoms."""
    G = int(match.flags.shape[0])
    if generated.flags.shape[0] != G:
        raise ValueError(f"{G} pairs against metrics of {generated.flags.shape[0]} generated crystals")
    ok = match.matched & generated.valid & generated.known
    count = lambda bit: int(((match.flags & bit) != 0).sum())  # noqa: E731
    return dict(num_pairs=G, num_matched=int(ok.sum()), match_rate=int(ok.sum()) / G if G else None,
                mean_rms=float(match.rms[ok].mean()) if ok.any() else None,
                num_composition_mismatch=count(COMPOSITION), num_match_search_limit=count(SEARCH_LIMIT),
                num_match_degenerate=count(DEGENERATE), num_too_large=count(TOO_LARGE))


def select_crystals(inputs, index):
    """The crystals `index` (in that order) of (frac_x, lattice, atomic_numbers, num_atoms) host arrays."""
    frac, lattice, z, na = inputs
    index = np.asarray(index, dtype=np.int64).reshape(-1)
    off = np.concatenate([[0], np.cumsum(na)]).astype(np.int64)
    atoms = np.concatenate([np.arange(off[i], off[i + 1]) for i in index]) if len(index) else np.zeros(0, np.int64)
    return frac[atoms], lattice[index], z[atoms], np.asarray(na)[index]


def check_source_index(source_index: Optional[np.ndarray], num_crystals: int, num_sources: int) -> np.ndarray:
    """source_index as int64 after checking it exists, has one entry per generated crystal and indexes the source
    data set (ValueError otherwise)."""
    if source_index is None:
        raise ValueError("the samples file has no source_index (write it with generate --compositions_from or "
                         "--structures_from)")
    idx = np.asarray(source_index).reshape(-1)
    if idx.shape[0] != num_crystals:
        raise ValueError(f"source_index has {idx.shape[0]} entries for {num_crystals} generated crystals")
    if not np.issubdtype(idx.dtype, np.integer):
        raise ValueError(f"source_index must hold integers, not {idx.dtype}")
    bad = (idx < 0) | (idx >= num_sources)
    if bad.any():
        raise ValueError(f"source_index {int(idx[bad][0])} is outside the reference data set of {num_sources} "
                         "crystals: --reference must be the files generate drew from")
    return idx.astype(np.int64)
