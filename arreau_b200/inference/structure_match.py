"""Match rate and RMSE of generated crystals against their source structures (crystal structure prediction), and
uniqueness and novelty of generated crystals, on the GPU.

    python -m arreau_b200.inference.crystal_metrics out/crystals.h5 --reference DATA --match
    python -m arreau_b200.inference.crystal_metrics out/crystals.h5 --reference TRAIN --unique_novel

`structure_match` pairs generated crystal i with source crystal i and runs `arreau_structure_match` (csrc/match.cu):
pymatgen's StructureMatcher(stol=0.5, ltol=0.3, angle_tol=10, scale=True, attempt_supercell=False).get_rms_dist as
DiffCSP calls it, without the primitive-cell reduction.  `match_summary` gives DiffCSP's match rate (matched and
structurally valid over all pairs) and the mean RMSE over the matched pairs.

`structure_fit_pairs` decides pymatgen's StructureMatcher(stol=0.3, ltol=0.2, angle_tol=5, scale=True,
attempt_supercell=False).fit on arbitrary pairs of crystals of two sets (`arreau_structure_fit_pairs`, the same
kernel), `unique_novel` builds group_structures and novelty against a reference on it, and `unique_novel_summary`
gives the counts and fractions.  The semantics, the deviations from pymatgen and the measured speed are in DESIGN.md
section 6."""
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


@dataclass
class FitPairs:
    """Per-pair results of structure_fit_pairs, numpy arrays of length P.  max_dist is normalised as in
    StructureMatch: the first value below stol when matched, else the smallest found (NaN without a candidate)."""
    matched: np.ndarray        # bool, fit(crystal index1[p] of set 1, crystal index2[p] of set 2)
    max_dist: np.ndarray
    num_mappings: np.ndarray   # int32, lattice mappings visited (all of them when not matched)
    flags: np.ndarray          # int32, MATCHED | COMPOSITION | DEGENERATE | SEARCH_LIMIT | TOO_LARGE


# pairs per launch of structure_fit_pairs: bounds the device output buffer of a chunk (16 bytes per pair)
MAX_CHUNK_PAIRS = 1 << 20


def _upload_used(inputs, na, off, index, dev):
    """The crystals of `inputs` that `index` names, Z-sorted, on `dev` as (frac, lattice, z, offset) tensors, and
    `index` renumbered into them (int32; an index outside the set becomes -1, which the kernel flags DEGENERATE)."""
    G = len(na)
    index = np.asarray(index, dtype=np.int64).reshape(-1)
    inside = (index >= 0) & (index < G)
    used = np.unique(index[inside])
    local = np.full(index.shape, -1, dtype=np.int32)
    local[inside] = np.searchsorted(used, index[inside])
    frac, lattice, z, _ = _sorted_by_z(inputs)
    o = np.zeros(len(used) + 1, dtype=np.int64)
    np.cumsum(na[used], out=o[1:])
    atoms = np.arange(o[-1], dtype=np.int64) + np.repeat(off[used] - o[:-1], na[used])
    frac, lattice, z, o = frac[atoms], lattice[used], z[atoms], o.astype(np.int32)
    tensors = (_rows_on(frac, 0, len(z), torch.float64, dev), _rows_on(lattice, 0, len(used), torch.float64, dev),
               _rows_on(z, 0, len(z), torch.int64, dev), _rows_on(o, 0, len(o), torch.int32, dev))
    return tensors, len(z), len(used), local


def structure_fit_pairs(set1, set2, index1, index2, stol: float = 0.3, ltol: float = 0.2, angle_tol: float = 5.0,
                        device="cuda", max_chunk_pairs: int = MAX_CHUNK_PAIRS) -> FitPairs:
    """fit(crystal index1[p] of set1, crystal index2[p] of set2) for every p, as pymatgen's StructureMatcher(stol,
    ltol, angle_tol, primitive_cell=False, scale=True, attempt_supercell=False).fit decides it (`arreau_structure_fit_pairs`,
    csrc/match.cu); set1's lattice is the one mapped.  Both sets are (frac_x, lattice, atomic_numbers, num_atoms) as
    `sample_inputs` / `dataset_inputs` return them, and may be the same object.  Only the crystals the pairs name are
    uploaded (Z-sorted); the pairs run in chunks of at most `max_chunk_pairs`, one device->host read each, and a
    pair's results do not depend on the chunking, the order or the other pairs.  An index outside its set gives
    DEGENERATE."""
    dev = _cuda_device(device, "structure_fit_pairs")
    for name, v in (("stol", stol), ("ltol", ltol), ("angle_tol", angle_tol)):
        if not (np.isfinite(v) and v > 0):
            raise ValueError(f"{name} must be finite and positive, got {v}")
    i1 = np.asarray(index1).reshape(-1)
    i2 = np.asarray(index2).reshape(-1)
    if i1.shape != i2.shape:
        raise ValueError(f"index1 has {i1.shape[0]} pairs, index2 {i2.shape[0]}")
    if any(x.size and not np.issubdtype(x.dtype, np.integer) for x in (i1, i2)):
        raise ValueError("index1 and index2 must hold integers")
    P = int(i1.shape[0])
    if P >= 2 ** 31:
        raise ValueError("at most 2^31 - 1 pairs")
    if P == 0:
        return FitPairs(matched=np.zeros(0, np.bool_), max_dist=np.zeros(0), num_mappings=np.zeros(0, np.int32),
                        flags=np.zeros(0, np.int32))
    na1, off1 = _check_inputs(*set1)
    na2, off2 = _check_inputs(*set2)
    t1, n1, g1, x1 = _upload_used(set1, na1, off1, i1, dev)
    t2, n2, g2, x2 = _upload_used(set2, na2, off2, i2, dev)
    x1 = _rows_on(x1, 0, P, torch.int32, dev)
    x2 = _rows_on(x2, 0, P, torch.int32, dev)

    def launch(p0, p1, outs, stream):
        _lib.call("arreau_structure_fit_pairs", *[t.data_ptr() for t in t1], n1, g1, *[t.data_ptr() for t in t2], n2,
                  g2, x1[p0:].data_ptr(), x2[p0:].data_ptr(), p1 - p0, float(stol), float(ltol), float(angle_tol),
                  *outs, stream)

    max_dist, num_mappings, flags = _run_chunked(np.arange(P + 1, dtype=np.int64), max_chunk_pairs,
                                                 (np.float64, np.int32, np.int32), launch, dev)
    return FitPairs(matched=(flags & MATCHED) != 0, max_dist=max_dist, num_mappings=num_mappings, flags=flags)


def composition_keys(atomic_numbers, num_atoms) -> list:
    """One hashable key per crystal: its exact multiset of Z (atom count included), as the bytes of its sorted
    atomic numbers.  With primitive_cell=False and no supercells, fit never holds between different keys."""
    z = np.asarray(atomic_numbers, dtype=np.int64).reshape(-1)
    na = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
    crystal = np.repeat(np.arange(len(na)), na)
    zs = z[np.lexsort((z, crystal))]
    off = np.concatenate([[0], np.cumsum(na)])
    return [zs[off[g]:off[g + 1]].tobytes() for g in range(len(na))]


def reduced_formula(key: bytes) -> tuple:
    """The reduced formula of a composition key: its (Z, count / gcd of the counts) pairs."""
    el, cnt = np.unique(np.frombuffer(key, dtype=np.int64), return_counts=True)
    d = np.gcd.reduce(cnt) if cnt.size else 1
    return tuple(zip(el.tolist(), (cnt // d).tolist()))


def _members(keys, select) -> dict:
    """key -> the indices i with select[i], ascending."""
    out = {}
    for i in np.nonzero(select)[0]:
        out.setdefault(keys[i], []).append(int(i))
    return out


def uniqueness_pairs(keys, considered):
    """(index1, index2) int64: every (j, i) of considered crystals j < i with equal keys."""
    firsts, seconds = [], []
    for m in _members(keys, considered).values():
        if len(m) > 1:
            a, b = np.triu_indices(len(m), 1)
            firsts.append(np.asarray(m)[a])
            seconds.append(np.asarray(m)[b])
    cat = lambda x: np.concatenate(x).astype(np.int64) if x else np.zeros(0, np.int64)  # noqa: E731
    return cat(firsts), cat(seconds)


def novelty_pairs(keys, considered, ref_keys):
    """(index1, index2) int64: every (i, r) of a considered crystal i and a reference crystal r with i's key."""
    ref = _members(ref_keys, np.ones(len(ref_keys), np.bool_))
    firsts, seconds = [], []
    for i in np.nonzero(considered)[0]:
        r = ref.get(keys[i])
        if r:
            firsts.append(np.full(len(r), i, np.int64))
            seconds.append(np.asarray(r, np.int64))
    cat = lambda x: np.concatenate(x).astype(np.int64) if x else np.zeros(0, np.int64)  # noqa: E731
    return cat(firsts), cat(seconds)


def resolve_groups(considered, index1, index2, matched) -> np.ndarray:
    """pymatgen's group_structures on a given fit relation: walking the considered crystals in order, crystal i joins
    the group of the earliest earlier representative r with fit(r, i) (pair (r, i) matched), else it is a
    representative.  Returns group[G], the representative's index (-1 where not considered).  Pairs (j, i) must have
    j < i; pairs that are not listed count as not matched."""
    considered = np.asarray(considered, np.bool_)
    group = np.where(considered, np.arange(len(considered)), -1)
    m = np.asarray(matched, np.bool_)
    j, i = np.asarray(index1, np.int64)[m], np.asarray(index2, np.int64)[m]
    if np.any(j >= i):
        raise ValueError("uniqueness pairs must have index1 < index2")
    order = np.lexsort((j, i))
    j, i = j[order], i[order]
    is_rep = considered.copy()
    p = 0
    while p < len(i):             # every i with a matched pair, ascending, its earlier partners ascending
        q = p
        while q < len(i) and i[q] == i[p]:
            q += 1
        for jj in j[p:q]:
            if is_rep[jj]:
                group[i[p]] = jj
                is_rep[i[p]] = False
                break
        p = q
    return group


@dataclass
class UniqueNovel:
    """Per generated crystal (length G): considered (structurally valid with known elements), group (index of its
    group's representative, -1 where not considered), unique (a representative), novel (no reference crystal fits;
    None without a reference), new_formula (its reduced formula does not occur in the reference; None without one);
    and the pairs evaluated with their results."""
    considered: np.ndarray
    group: np.ndarray
    unique: np.ndarray
    novel: Optional[np.ndarray]
    new_formula: Optional[np.ndarray]
    uniqueness_pairs: tuple    # (index1, index2) into the generated crystals
    uniqueness_fit: FitPairs
    novelty_pairs: tuple       # (generated index, reference index)
    novelty_fit: Optional[FitPairs]


def unique_novel(gen_inputs, generated: CrystalMetrics, ref_inputs=None, stol: float = 0.3, ltol: float = 0.2,
                 angle_tol: float = 5.0, device="cuda", max_chunk_pairs: int = MAX_CHUNK_PAIRS) -> UniqueNovel:
    """Uniqueness and novelty of generated crystals (frac_x, lattice, atomic_numbers, num_atoms) with their
    crystal_metrics, against the reference data set `ref_inputs` (the training data; optional).  Only crystals that
    are structurally valid with known elements are considered.  The key of a crystal is its exact multiset of Z.
    Uniqueness is pymatgen's group_structures: fit runs on every pair (j, i) of considered crystals j < i with equal
    keys, in one chunked launch, and resolve_groups applies its greedy rule; this is a superset of the pairs
    group_structures evaluates and gives its groups exactly.  Crystal i is novel when it is considered and fit(i, r)
    holds for no reference crystal r with its key (a second launch)."""
    G = int(np.asarray(gen_inputs[3]).reshape(-1).shape[0])
    if generated.flags.shape[0] != G:
        raise ValueError(f"{G} generated crystals against metrics of {generated.flags.shape[0]}")
    considered = generated.valid & generated.known
    keys = composition_keys(gen_inputs[2], gen_inputs[3])
    kw = dict(stol=stol, ltol=ltol, angle_tol=angle_tol, device=device, max_chunk_pairs=max_chunk_pairs)
    up = uniqueness_pairs(keys, considered)
    ufit = structure_fit_pairs(gen_inputs, gen_inputs, *up, **kw)
    group = resolve_groups(considered, *up, ufit.matched)
    unique = considered & (group == np.arange(G))
    novel = new_formula = nfit = None
    npairs = (np.zeros(0, np.int64), np.zeros(0, np.int64))
    if ref_inputs is not None:
        ref_keys = composition_keys(ref_inputs[2], ref_inputs[3])
        npairs = novelty_pairs(keys, considered, ref_keys)
        nfit = structure_fit_pairs(gen_inputs, ref_inputs, *npairs, **kw)
        fits_ref = np.zeros(G, np.bool_)
        fits_ref[npairs[0][nfit.matched]] = True
        novel = considered & ~fits_ref
        ref_formulas = {reduced_formula(k) for k in set(ref_keys)}
        new = {k: reduced_formula(k) not in ref_formulas for k in set(keys)}
        new_formula = considered & np.array([new[k] for k in keys], np.bool_).reshape(-1)
    return UniqueNovel(considered=considered, group=group, unique=unique, novel=novel, new_formula=new_formula,
                       uniqueness_pairs=up, uniqueness_fit=ufit, novelty_pairs=npairs, novelty_fit=nfit)


def unique_novel_summary(un: UniqueNovel) -> dict:
    """JSON-ready summary (None where a set is empty): num_unique, num_novel and num_unique_novel with their
    fractions over all generated crystals (as match_rate), num_new_formula (considered crystals whose reduced formula
    the reference does not hold: novel under any matcher settings), num_fit_pairs, and the counts of pairs flagged
    SEARCH_LIMIT, DEGENERATE or TOO_LARGE (counted as not matched).  Without a reference only the uniqueness keys."""
    G = int(un.considered.shape[0])
    frac = lambda k: k / G if G else None  # noqa: E731
    fits = [un.uniqueness_fit] + ([un.novelty_fit] if un.novelty_fit is not None else [])
    count = lambda bit: int(sum(((f.flags & bit) != 0).sum() for f in fits))  # noqa: E731
    out = dict(num_considered=int(un.considered.sum()), num_unique=int(un.unique.sum()),
               frac_unique=frac(int(un.unique.sum())))
    if un.novel is not None:
        both = int((un.unique & un.novel).sum())
        out.update(num_novel=int(un.novel.sum()), frac_novel=frac(int(un.novel.sum())), num_unique_novel=both,
                   frac_unique_novel=frac(both), num_new_formula=int(un.new_formula.sum()))
    out.update(num_fit_pairs=int(sum(len(f.flags) for f in fits)), num_fit_search_limit=count(SEARCH_LIMIT),
               num_fit_degenerate=count(DEGENERATE), num_fit_too_large=count(TOO_LARGE))
    return out


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
