"""arreau_structure_fit_pairs / inference.structure_match.unique_novel on the GPU against the numpy fit oracle of
test_unique_novel_host.py: about 500 pairs (transformed and displaced copies, random positions, high-symmetry cells),
the relation to structure_match, independence of batch, order and chunking, an out-of-range index, a constructed set
with a known answer, group_structures on a few hundred crystals, and crystal_metrics --unique_novel end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_structure_match import _alexandria, _high_symmetry, _pack
from test_structure_match_host import DEGENERATE, MATCHED, transformed_copy
from test_unique_novel_host import _crystal, _metrics, fit_pair, fit_pairs, group_structures, groups_of

STOL = 0.3


def _same_composition(num, per, lo, hi, seed):
    """`num` compositions of Alexandria-shaped crystals with `per` structures each (random positions, the cell
    perturbed), listed composition by composition: [(frac, lattice, z)]."""
    rng = np.random.default_rng(seed)
    out = []
    for f, L, z in _alexandria(num, lo, hi, seed=seed):
        for _ in range(per):
            out.append((rng.random((len(z), 3)), L @ np.diag(1 + 0.05 * rng.standard_normal(3)), z))
    return out


@pytest.fixture(scope="module")
def fit_cases():
    """~500 pairs (index1, index2) into two sets and the oracle's results, none within 1e-9 of stol."""
    rng = np.random.default_rng(0)
    first, second = [], []
    for k, c in enumerate(_alexandria(320, 1, 24, seed=11)):
        first.append(transformed_copy(*c, rng, sigma=(0.0, 0.02, 0.06, 0.2)[k % 4]))
        second.append(c)
    for c in _alexandria(100, 1, 24, seed=12):
        n = len(c[2])
        first.append((rng.random((n, 3)), c[1] @ np.diag(1 + 0.05 * rng.standard_normal(3)), c[2][rng.permutation(n)]))
        second.append(c)
    for k in range(80):
        c = _high_symmetry()[k % 5]
        first.append(transformed_copy(np.asarray(c[0], np.float64), c[1], np.asarray(c[2]), rng,
                                      sigma=(0.0, 0.02, 0.1, 0.3)[(k // 5) % 4]))
        second.append(c)
    P = len(first)
    p1, p2 = rng.permutation(P), rng.permutation(P)          # pair p is first[p] against second[p], stored shuffled
    set1, set2 = _pack([first[i] for i in p1]), _pack([second[i] for i in p2])
    index1, index2 = np.argsort(p1), np.argsort(p2)
    expect = fit_pairs(set1, set2, index1, index2)
    keep = ~(np.abs(expect["max_dist"] - STOL) < 1e-9)
    return set1, set2, index1[keep], index2[keep], {k: v[keep] for k, v in expect.items()}


@pytest.mark.gpu
def test_fit_kernel_matches_the_oracle(device, fit_cases):
    from arreau_b200.inference.structure_match import structure_fit_pairs
    set1, set2, i1, i2, expect = fit_cases
    r = structure_fit_pairs(set1, set2, i1, i2, device=device)
    np.testing.assert_array_equal(r.flags, expect["flags"])
    matched = (r.flags & MATCHED) != 0
    assert np.all(r.max_dist[matched] < STOL)
    un = ~matched
    np.testing.assert_array_equal(r.num_mappings[un], expect["num_mappings"][un])
    a, b = r.max_dist[un], expect["max_dist"][un]
    assert np.array_equal(np.isnan(a), np.isnan(b))
    fin = np.isfinite(b)
    assert np.abs(a[fin] - b[fin]).max(initial=0) <= 1e-9, np.abs(a[fin] - b[fin]).max()
    assert matched.sum() > 200 and un.sum() > 50 and r.num_mappings.max() >= 48
    print(f"{len(r.flags)} pairs: {int(matched.sum())} matched, mappings visited mean {r.num_mappings.mean():.1f} "
          f"(matched {r.num_mappings[matched].mean():.1f}), max {int(r.num_mappings.max())}")


@pytest.mark.gpu
def test_fit_implies_an_rms_match(device, fit_cases):
    from arreau_b200.inference.structure_match import select_crystals, structure_fit_pairs, structure_match
    set1, set2, i1, i2, _ = fit_cases
    r = structure_fit_pairs(set1, set2, i1, i2, device=device)
    m = structure_match(select_crystals(set1, i1), select_crystals(set2, i2), stol=STOL, ltol=0.2, angle_tol=5.0,
                        device=device)
    matched = (r.flags & MATCHED) != 0
    assert np.all(m.matched[matched])
    assert np.all(m.rms[matched] <= r.max_dist[matched] + 1e-12)
    np.testing.assert_array_equal(r.num_mappings[~matched], m.num_mappings[~matched])
    np.testing.assert_array_equal(r.flags & ~MATCHED, m.flags & ~MATCHED)
    assert np.all(r.num_mappings[matched] <= m.num_mappings[matched])
    print(f"fit {int(matched.sum())}, rms {int(m.matched.sum())} of {len(r.flags)}; mappings visited "
          f"{int(r.num_mappings.sum())} against {int(m.num_mappings.sum())}")


@pytest.mark.gpu
def test_fit_results_do_not_depend_on_batch_or_order(device, fit_cases):
    from arreau_b200.inference.structure_match import structure_fit_pairs
    set1, set2, i1, i2, _ = fit_cases
    whole = structure_fit_pairs(set1, set2, i1, i2, device=device)
    keys = ("max_dist", "num_mappings", "flags")
    rng = np.random.default_rng(1)
    # shuffled and repeated indices
    sel = np.concatenate([rng.permutation(len(i1)), rng.integers(0, len(i1), 200)])
    r = structure_fit_pairs(set1, set2, i1[sel], i2[sel], device=device)
    for k in keys:
        assert getattr(r, k).tobytes() == getattr(whole, k)[sel].tobytes(), k
    # one set holding both: set 1 is set 2
    both = tuple(np.concatenate([a, b]) for a, b in zip(set1, set2))
    r = structure_fit_pairs(both, both, i1, i2 + len(set1[3]), device=device)
    for k in keys:
        assert getattr(r, k).tobytes() == getattr(whole, k).tobytes(), k
    # other chunk sizes
    for chunk in (1, 37):
        r = structure_fit_pairs(set1, set2, i1, i2, device=device, max_chunk_pairs=chunk)
        for k in keys:
            assert getattr(r, k).tobytes() == getattr(whole, k).tobytes(), (k, chunk)


@pytest.mark.gpu
def test_out_of_range_index_is_degenerate(device, fit_cases):
    from arreau_b200.inference.structure_match import structure_fit_pairs
    set1, set2, i1, i2, _ = fit_cases
    G1, G2 = len(set1[3]), len(set2[3])
    r = structure_fit_pairs(set1, set2, [-1, G1, 0, i1[0], 2 ** 31 - 1], [0, 0, -5, G2, i2[0]], device=device)
    assert r.flags.tolist() == [DEGENERATE] * 5
    assert np.isnan(r.max_dist).all() and (r.num_mappings == 0).all()
    assert len(structure_fit_pairs(set1, set2, [], [], device=device).flags) == 0


@pytest.mark.gpu
def test_known_groups_and_novelty(device):
    from arreau_b200.inference.structure_match import unique_novel, unique_novel_summary
    rng = np.random.default_rng(5)
    bases = _same_composition(10, 3, 6, 12, seed=13)          # 30 bases, three per composition
    family = []
    for b in range(len(bases)):
        family += [b] * (1 + b % 3)                           # one to three members each
    family = np.array(family)[rng.permutation(len(family))]
    gen = [transformed_copy(*bases[b], rng, sigma=(0.0, 0.02)[k % 2]) for k, b in enumerate(family)]
    in_ref = np.arange(len(bases)) % 2 == 0                   # half of the bases, transformed again
    ref = [transformed_copy(*bases[b], rng, sigma=0.02) for b in np.nonzero(in_ref)[0]]
    g, r = _pack(gen), _pack(ref)
    un = unique_novel(g, _metrics(np.ones(len(gen), np.int32)), r, device=device)
    expect = {}
    for i, b in enumerate(family):
        expect.setdefault(int(b), []).append(i)
    assert groups_of(un.group) == sorted(expect.values())
    np.testing.assert_array_equal(un.novel, ~in_ref[family])
    assert not un.new_formula.any()
    s = unique_novel_summary(un)
    assert s["num_unique"] == 30 and s["num_novel"] == int((~in_ref[family]).sum()) and s["num_unique_novel"] == 15
    assert s["num_fit_search_limit"] == s["num_fit_degenerate"] == s["num_fit_too_large"] == 0


@pytest.mark.gpu
def test_unique_novel_is_group_structures(device):
    from arreau_b200.inference.structure_match import composition_keys, unique_novel
    rng = np.random.default_rng(6)
    pool = _same_composition(16, 1, 1, 8, seed=14)            # small crystals: random ones often fit
    crystals = []
    for k in range(240):
        if k >= 16 and rng.random() < 0.4:                    # a copy of an earlier crystal
            crystals.append(transformed_copy(*crystals[int(rng.integers(0, k))], rng, sigma=0.02))
        else:
            f, L, z = pool[int(rng.integers(0, len(pool)))]
            crystals.append((rng.random((len(z), 3)), L @ np.diag(1 + 0.05 * rng.standard_normal(3)), z))
    ref_crystals = [transformed_copy(*crystals[int(i)], rng, sigma=0.02) for i in rng.integers(0, 240, 20)]
    ref_crystals += [(rng.random((len(c[2]), 3)), c[1], c[2]) for c in pool]
    g, r = _pack(crystals), _pack(ref_crystals)
    flags = np.where(rng.random(240) < 0.9, 1, 0).astype(np.int32)          # some crystals not valid
    un = unique_novel(g, _metrics(flags), r, device=device)
    keys = composition_keys(g[2], g[3])
    fit = lambda a, b: fit_pair(*_crystal(g, a), *_crystal(g, b))["flags"] == MATCHED  # noqa: E731
    expect = group_structures(flags == 1, keys, fit)
    assert groups_of(un.group) == sorted(expect)
    rk = composition_keys(r[2], r[3])
    novel = np.array([flags[i] == 1 and not any(fit_pair(*_crystal(g, i), *_crystal(r, j))["flags"] == MATCHED
                                                for j in range(len(rk)) if rk[j] == keys[i]) for i in range(240)])
    np.testing.assert_array_equal(un.novel, novel)
    sizes = [len(x) for x in expect]
    assert max(sizes) > 3 and len(expect) > 40 and 0 < novel.sum() < (flags == 1).sum()
    print(f"{len(expect)} groups (largest {max(sizes)}), {int(novel.sum())} novel, "
          f"{len(un.uniqueness_fit.flags)} + {len(un.novelty_fit.flags)} pairs")


@pytest.mark.gpu
def test_cli_unique_novel_end_to_end(device, tmp_path):
    from arreau_b200.diffusion.diffusion_loss import SampleResult
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    from arreau_b200.inference.crystal_metrics import crystal_metrics, dataset_inputs
    from arreau_b200.inference.process_generated_crystals import save_sample_results_to_hdf5
    from arreau_b200.inference.structure_match import select_crystals, unique_novel, unique_novel_summary
    rng = np.random.default_rng(7)
    data_crystals = _same_composition(10, 3, 2, 10, seed=15)
    data = save_dataset_npz(str(tmp_path / "data"), [c[2] for c in data_crystals],
                            np.stack([c[1] for c in data_crystals]), [c[0] for c in data_crystals])
    ref = dataset_inputs(CrystalDataset([data]))
    index = rng.integers(0, 30, 24)
    src = select_crystals(ref, index)
    gen = [transformed_copy(*_crystal(src, i), rng, sigma=0.02) for i in range(12)]
    gen += [(rng.random((len(c[2]), 3)), c[1], c[2]) for c in _same_composition(12, 1, 2, 10, seed=16)]
    g = _pack(gen)
    res = SampleResult(frac_x=g[0], lattice=g[1], atomic_numbers=g[2], num_atoms=g[3],
                       idx_start=np.concatenate([[0], np.cumsum(g[3])[:-1]]))
    out = save_sample_results_to_hdf5(res, str(tmp_path / "crystals.npz"))
    js = str(tmp_path / "metrics.json")
    r = subprocess.run([sys.executable, "-m", "arreau_b200.inference.crystal_metrics", out, "--reference", data,
                        "--unique_novel", "--json", js], cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    with open(js) as fh:
        got = json.load(fh)
    expect = unique_novel_summary(unique_novel(g, crystal_metrics(*g, device=device), ref, device=device))
    for k, v in expect.items():
        assert got[k] == v, k
    for k in ("frac_unique", "frac_novel", "frac_unique_novel", "num_new_formula", "num_fit_pairs", "frac_valid"):
        assert k in got
    assert got["num_fit_pairs"] > 0
