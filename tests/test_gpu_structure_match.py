"""arreau_structure_match / inference.structure_match on the GPU against the numpy oracle of
test_structure_match_host.py: about 500 pairs (transformed and displaced copies, random positions, high-symmetry cells),
batch independence, edge cases and crystal_metrics --match end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_structure_match_host import (COMPOSITION, DEGENERATE, MATCHED, SEARCH_LIMIT, TOO_LARGE, match_pairs,
                                       transformed_copy, wrap)

ELEMENTS = np.array([3, 8, 12, 26, 29])


def _pack(crystals):
    """[(frac[n,3], lattice[3,3], z[n])] -> (frac, lattice, z, num_atoms)."""
    return (np.concatenate([np.asarray(c[0], np.float64).reshape(-1, 3) for c in crystals]),
            np.stack([np.asarray(c[1], np.float64) for c in crystals]),
            np.concatenate([np.asarray(c[2], np.int64).reshape(-1) for c in crystals]),
            np.array([len(c[2]) for c in crystals], np.int64))


def _alexandria(num, lo, hi, seed):
    """Alexandria-shaped crystals (synthetic.make_crystals) over five elements: [(frac, lattice, z)]."""
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R
    cr = make_crystals(num, lo, hi, seed=seed)
    lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
    off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
    return [(cr.frac[off[g]:off[g + 1]], lat[g], ELEMENTS[cr.types[off[g]:off[g + 1]] % 5]) for g in range(num)]


def _high_symmetry():
    a = 3.6
    hexa = np.array([[a, 0, 0], [-a / 2, a * np.sqrt(3) / 2, 0], [0, 0, 1.63 * a]])
    return [(np.zeros((1, 3)), np.eye(3) * 2.9, [26]),                                          # simple cubic
            (np.array([[0, 0, 0], [0.5, 0.5, 0.5]]), np.eye(3) * 4.1, [17, 55]),                 # CsCl
            (np.array([[1 / 3, 2 / 3, 0.25], [2 / 3, 1 / 3, 0.75]]), hexa, [12, 12]),            # hcp
            (np.array([[0, 0, 0], [0, .5, .5], [.5, 0, .5], [.5, .5, 0]]), np.eye(3) * a, [29] * 4),  # fcc conv.
            (np.array([[0, 0, 0], [.5, .5, .5], [0, 0, .5], [.5, .5, 0], [0, .5, 0], [.5, 0, .5], [.5, 0, 0],
                       [0, .5, .5]]), np.eye(3) * 5.64, [11] * 4 + [17] * 4)]                    # rock salt conv.


@pytest.fixture(scope="module")
def pairs():
    """~500 (generated, source) pairs and the oracle's results, none within 1e-9 of stol."""
    rng = np.random.default_rng(0)
    gen, ref = [], []
    for k, c in enumerate(_alexandria(320, 1, 24, seed=1)):
        gen.append(transformed_copy(*c, rng, sigma=(0.0, 0.02, 0.1, 0.3)[k % 4]))
        ref.append(c)
    for c in _alexandria(100, 1, 24, seed=2):            # the same kind of compositions at random positions
        n = len(c[2])
        gen.append((rng.random((n, 3)), c[1] @ np.diag(1 + 0.05 * rng.standard_normal(3)), c[2][rng.permutation(n)]))
        ref.append(c)
    for k in range(80):
        c = _high_symmetry()[k % 5]
        gen.append(transformed_copy(np.asarray(c[0], np.float64), c[1], np.asarray(c[2]), rng,
                                    sigma=(0.0, 0.03, 0.15, 0.4)[(k // 5) % 4]))
        ref.append(c)
    g, r = _pack(gen), _pack(ref)
    expect = match_pairs(g, r)
    near = np.abs(expect["rms"] - 0.5) < 1e-9
    if near.any():
        keep = np.nonzero(~near)[0]
        from arreau_b200.inference.structure_match import select_crystals
        g, r = select_crystals(g, keep), select_crystals(r, keep)
        expect = {k: v[keep] for k, v in expect.items()}
    return g, r, expect


def _assert_agrees(m, expect):
    np.testing.assert_array_equal(m.flags, expect["flags"])
    np.testing.assert_array_equal(m.num_mappings, expect["num_mappings"])
    for k in ("rms", "max_dist"):
        a, b = getattr(m, k), expect[k]
        assert np.array_equal(np.isnan(a), np.isnan(b)), k
        fin = np.isfinite(b)
        err = np.abs(a[fin] - b[fin])
        assert err.max(initial=0) <= 1e-9, (k, err.max(), np.nonzero(np.abs(a - b) > 1e-9)[0][:10])


@pytest.mark.gpu
def test_kernel_matches_the_oracle(device, pairs):
    from arreau_b200.inference.structure_match import structure_match
    g, r, expect = pairs
    m = structure_match(g, r, device=device)
    _assert_agrees(m, expect)
    matched = (m.flags & MATCHED) != 0
    assert matched.sum() > 200 and (~matched).sum() > 50 and m.num_mappings.max() >= 48
    print(f"{len(m.flags)} pairs: {int(matched.sum())} matched, num_mappings up to {int(m.num_mappings.max())}")


@pytest.mark.gpu
def test_results_do_not_depend_on_batch_or_order(device, pairs):
    from arreau_b200.inference.structure_match import select_crystals, structure_match
    g, r, _ = pairs
    whole = structure_match(g, r, device=device)
    G = len(g[3])
    perm = np.random.default_rng(1).permutation(G)
    got = {k: np.empty_like(getattr(whole, k)) for k in ("rms", "max_dist", "num_mappings", "flags")}
    for part in np.array_split(perm, (G + 16) // 17):
        m = structure_match(select_crystals(g, part), select_crystals(r, part), device=device)
        for k in got:
            got[k][part] = getattr(m, k)
    chunked = structure_match(g, r, device=device, max_chunk_atoms=97)
    for k, v in got.items():
        assert v.tobytes() == getattr(whole, k).tobytes(), k
        assert getattr(chunked, k).tobytes() == getattr(whole, k).tobytes(), k


@pytest.mark.gpu
def test_edge_cases(device):
    from arreau_b200.inference.structure_match import structure_match
    rng = np.random.default_rng(4)
    big = _alexandria(1, 236, None, seed=5)[0]
    over = _alexandria(1, 257, None, seed=6)[0]
    cube = (rng.random((3, 3)), np.eye(3) * 4.0, [8, 8, 26])
    flat = (cube[0], np.array([[4.0, 0, 0], [0, 4.0, 0], [4.0, 4.0, 0]]), cube[2])
    nan = (cube[0], np.full((3, 3), np.nan), cube[2])
    needle = (cube[0], np.diag([0.4, 0.4, 400.0]), cube[2])         # same volume as the cube, 1000 times longer
    gen = [transformed_copy(*big, rng, sigma=0.02), over, cube, flat, cube, cube, cube]
    ref = [big, over, cube, cube, nan, needle, (cube[0], cube[1], [8, 8, 27])]
    g, r = _pack(gen), _pack(ref)
    m = structure_match(g, r, device=device)
    expect = match_pairs(g, r)
    _assert_agrees(m, expect)
    assert m.flags[0] == MATCHED and m.flags[1] == TOO_LARGE and m.flags[2] == MATCHED
    assert m.flags[3] == DEGENERATE and m.flags[4] == DEGENERATE and m.flags[5] == SEARCH_LIMIT
    assert m.flags[6] == COMPOSITION and np.isnan(m.rms[6]) and m.num_mappings[6] == 0


@pytest.mark.gpu
def test_cli_match_end_to_end(device, tmp_path):
    from arreau_b200.diffusion.diffusion_loss import SampleResult
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    from arreau_b200.inference.crystal_metrics import crystal_metrics, dataset_inputs
    from arreau_b200.inference.process_generated_crystals import save_sample_results_to_hdf5
    from arreau_b200.inference.structure_match import select_crystals
    rng = np.random.default_rng(7)
    data_crystals = _alexandria(30, 2, 12, seed=8)
    data = save_dataset_npz(str(tmp_path / "data"), [c[2] for c in data_crystals], np.stack([c[1] for c in data_crystals]),
                            [c[0] for c in data_crystals])
    ref_all = dataset_inputs(CrystalDataset([data]))
    index = rng.integers(0, 30, 24)
    src = select_crystals(ref_all, index)
    off = np.concatenate([[0], np.cumsum(src[3])])
    gen = [transformed_copy(src[0][off[i]:off[i + 1]], src[1][i], src[2][off[i]:off[i + 1]], rng, sigma=0.05)
           for i in range(len(index))]
    f, lat, z = gen[5]
    gen[5] = (f, lat, np.where(np.arange(len(z)) == 0, 2001, z))   # one atom left in the mask state
    g = _pack(gen)
    res = SampleResult(frac_x=g[0], lattice=g[1], atomic_numbers=g[2], num_atoms=g[3],
                       idx_start=np.concatenate([[0], np.cumsum(g[3])[:-1]]))
    out = save_sample_results_to_hdf5(res, str(tmp_path / "crystals.npz"), {"source_index": index})
    js = str(tmp_path / "metrics.json")
    r = subprocess.run([sys.executable, "-m", "arreau_b200.inference.crystal_metrics", out, "--reference", data,
                        "--match", "--json", js], cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    with open(js) as fh:
        got = json.load(fh)
    expect = match_pairs(g, src)
    metrics = crystal_metrics(*g, device=device)
    ok = ((expect["flags"] & MATCHED) != 0) & metrics.valid & metrics.known
    assert got["num_pairs"] == 24 and got["num_composition_mismatch"] == 1 and expect["flags"][5] == COMPOSITION
    assert got["num_matched"] == int(ok.sum()) and got["match_rate"] == int(ok.sum()) / 24 and ok.sum() > 0
    assert abs(got["mean_rms"] - expect["rms"][ok].mean()) <= 1e-9
    assert "frac_valid" in got and "w1_density" in got
