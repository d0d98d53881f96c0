"""Crystal quality metrics (arreau_crystal_metrics / inference.crystal_metrics) and generation with a data set's atom
counts (generate --num_atoms_from).  The numpy oracle below is independent of the kernel's method: it searches the
unreduced basis, over the image box that the bound |df_i + k_i| <= R |r_i| gives with R from the k = 0 image."""
import ctypes as C
import itertools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

AMU = 1.66053906660


# ---- numpy oracle ---------------------------------------------------------------------------------------------------
def _brute_min_dist(f, L, widen=0, max_images=2_000_000):
    """Exact minimum-image distance over distinct pairs by brute force in the given basis."""
    i, j = np.triu_indices(len(f), 1)
    df = f[j] - f[i]
    R = np.sqrt(((df @ L) ** 2).sum(1)).min()
    r = np.linalg.norm(np.linalg.inv(L), axis=0)          # columns of L^-1
    lo = np.floor((-df).min(0) - R * r) - widen
    hi = np.ceil((-df).max(0) + R * r) + widen
    axes = [np.arange(a, b + 1) for a, b in zip(lo, hi)]
    assert np.prod([len(a) for a in axes]) <= max_images, "oracle image box too large"
    ks = np.array(list(itertools.product(*axes)), dtype=np.float64)
    best = np.inf
    for c in range(0, len(ks), max(1, 200_000 // len(df))):
        d = (df[:, None, :] + ks[None, c:c + max(1, 200_000 // len(df))]) @ L
        best = min(best, float(np.sqrt((d * d).sum(-1)).min()))
    return best


def oracle(frac, lattice, z, num_atoms, min_dist=0.5, min_volume=0.1):
    from arreau_b200.tools.atomic_number_table import ATOMIC_MASS
    mass = np.array(ATOMIC_MASS)
    off = np.concatenate([[0], np.cumsum(num_atoms)])
    G = len(num_atoms)
    out = dict(volume=np.empty(G), min_dist=np.empty(G), density=np.empty(G), num_elements=np.zeros(G, np.int32),
               flags=np.zeros(G, np.int32), volume_scale=np.empty(G), mass=np.empty(G))
    for g in range(G):
        f, L, zz = frac[off[g]:off[g + 1]], lattice[g], z[off[g]:off[g + 1]]
        with np.errstate(invalid="ignore"):
            vol = abs(np.linalg.det(L)) if np.isfinite(L).all() else np.nan
        known = (zz >= 1) & (zz <= len(mass))
        degenerate = not (np.isfinite(L).all() and np.isfinite(f).all() and vol >= min_volume)
        md = np.nan if degenerate else (np.inf if len(f) < 2 else _brute_min_dist(f, L))
        out["volume"][g] = vol
        out["min_dist"][g] = md
        out["mass"][g] = mass[zz - 1].sum() if known.all() else np.nan
        with np.errstate(divide="ignore", invalid="ignore"):
            out["density"][g] = out["mass"][g] * AMU / vol
        out["volume_scale"][g] = np.prod(np.linalg.norm(L, axis=1))
        out["num_elements"][g] = len(set(zz[known].tolist()))
        out["flags"][g] = (1 if (not degenerate and md >= min_dist) else 0) | (0 if known.all() else 2) | \
            (4 if degenerate else 0)
    return out


def _pack(crystals):
    """[(frac[n,3], lattice[3,3], z[n])] -> flat inputs."""
    frac = np.concatenate([np.asarray(c[0], np.float64).reshape(-1, 3) for c in crystals])
    lat = np.stack([np.asarray(c[1], np.float64) for c in crystals])
    z = np.concatenate([np.asarray(c[2], np.int64).reshape(-1) for c in crystals])
    na = np.array([len(np.asarray(c[2]).reshape(-1)) for c in crystals], np.int64)
    return frac, lat, z, na


def _skewed_cells(n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        L = np.diag(rng.uniform(2.0, 6.0, 3))
        L[1, 0] += rng.integers(-4, 5) * L[0, 0] + rng.uniform(-1, 1)
        L[2, :2] += rng.integers(-3, 4, 2) * np.array([L[0, 0], L[1, 1]]) + rng.uniform(-1, 1, 2)
        m = int(rng.integers(2, 6))
        out.append((rng.random((m, 3)), L, rng.integers(1, 104, m)))
    return out


def _assert_matches_oracle(m, ref):
    """flags and element counts exact; min_dist and density within 1e-12 relative.  The volume is a determinant: where
    it cancels (flat cells) its error is relative to the product of the row lengths, and the density is checked
    against the kernel's own volume."""
    np.testing.assert_array_equal(m.flags & ~8, ref["flags"])      # the oracle has no extended-search bit
    np.testing.assert_array_equal(m.num_elements, ref["num_elements"])
    with np.errstate(divide="ignore", invalid="ignore"):
        density = ref["mass"] * AMU / m.volume
    for k, a, b in (("volume", m.volume, ref["volume"]), ("min_dist", m.min_dist, ref["min_dist"]),
                    ("density", m.density, density)):
        assert np.array_equal(np.isnan(a), np.isnan(b)), k
        assert np.array_equal(np.isinf(a), np.isinf(b)), k
        fin = np.isfinite(b)
        atol = 1e-14 * ref["volume_scale"][fin] if k == "volume" else 0.0
        assert np.all(np.abs(a[fin] - b[fin]) <= 1e-12 * np.abs(b[fin]) + atol), k


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_oracle_agrees_with_a_wider_brute_force_on_skewed_cells():
    for f, L, _ in _skewed_cells(40, seed=1):
        assert _brute_min_dist(f, L) == _brute_min_dist(f, L, widen=3)


def test_atomic_mass_table():
    from arreau_b200.tools.atomic_number_table import ATOMIC_MASS, ATOMIC_NUMBER
    assert len(ATOMIC_MASS) == 103 == len(ATOMIC_NUMBER)
    spot = dict(H=1.008, C=12.011, O=15.999, Fe=55.845, U=238.029)
    for s, m in spot.items():
        assert round(ATOMIC_MASS[ATOMIC_NUMBER[s] - 1], 3) == m, s
    assert all(m > 0 for m in ATOMIC_MASS)


def _metrics(**kw):
    from arreau_b200.inference.crystal_metrics import CrystalMetrics
    return CrystalMetrics(**{k: np.asarray(v) for k, v in kw.items()})


def test_summarize_w1_and_exclusions():
    from scipy.stats import wasserstein_distance
    from arreau_b200.inference.crystal_metrics import summarize
    # flags: valid, valid, invalid, valid + unknown element, degenerate
    gen = _metrics(num_atoms=[4, 6, 2, 3, 5], volume=[50., 60., 20., 30., 0.],
                   min_dist=[1.2, 0.9, 0.3, 1.1, np.nan], density=[3.0, 4.5, 2.0, np.nan, np.inf],
                   num_elements=[2, 3, 1, 1, 2], flags=np.array([1, 1, 0, 3, 4], np.int32))
    ref = _metrics(num_atoms=[4, 8, 3], volume=[40., 70., 25.], min_dist=[1.5, 1.4, 2.0], density=[3.5, 5.0, np.nan],
                   num_elements=[2, 4, 1], flags=np.array([1, 1, 3], np.int32))
    s = summarize(gen, ref)
    assert (s["num_crystals"], s["num_valid"], s["num_unknown_element"], s["num_degenerate"]) == (5, 3, 1, 1)
    assert s["frac_valid"] == 0.6 and s["frac_degenerate"] == 0.2 and s["frac_unknown_element"] == 0.2
    assert s["min_dist_p50"] == np.percentile([1.2, 0.9, 0.3, 1.1], 50)
    assert s["mean_density"] == 3.75 and s["mean_num_elements"] == 2.5
    assert s["w1_density"] == wasserstein_distance([3.0, 4.5], [3.5, 5.0])
    assert s["w1_num_elements"] == wasserstein_distance([2, 3], [2, 4])
    assert s["w1_num_atoms"] == wasserstein_distance([4, 6, 2, 3, 5], [4, 8, 3])
    assert s["reference_frac_valid"] == 1.0 and s["reference_num_crystals"] == 3
    json.dumps(s)
    assert "w1_density" not in summarize(gen)
    empty = summarize(_metrics(num_atoms=[3], volume=[0.], min_dist=[np.nan], density=[np.inf], num_elements=[1],
                               flags=np.array([4], np.int32)), ref)
    assert empty["w1_density"] is None and empty["mean_density"] is None and empty["min_dist_p1"] is None


def test_metrics_entry_point_argument_validation():
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p)
    assert lib.arreau_crystal_metrics(None, None, None, None, 0, 0, None, 103, 0.5, 0.1, *([None] * 5), None) == 0
    assert lib.arreau_crystal_metrics(p, None, p, p, 4, 1, p, 103, 0.5, 0.1, *([p] * 5), None) == -4
    assert lib.arreau_crystal_metrics(p, p, p, p, 4, 1, p, 103, 0.5, 0.1, p, p, p, None, p, None) == -4
    assert lib.arreau_crystal_metrics(p, p, p, p, 4, -1, p, 103, 0.5, 0.1, *([p] * 5), None) == -1
    assert lib.arreau_crystal_metrics(p, p, p, p, -4, 1, p, 103, 0.5, 0.1, *([p] * 5), None) == -1
    assert lib.arreau_crystal_metrics(p, p, p, p, 4, 1, p, -1, 0.5, 0.1, *([p] * 5), None) == -1
    assert lib.arreau_crystal_metrics(p, p, p, p, 4, 1, p, 103, float("nan"), 0.1, *([p] * 5), None) == -1


def test_num_atoms_draw_is_seeded_and_independent_of_the_world_size():
    from arreau_b200.distributed import shard_range
    from arreau_b200.generate import draw_num_atoms
    data = np.array([4, 4, 4, 8, 8, 20, 1, 4, 8, 236])
    a = draw_num_atoms(data, 1001, seed=3)
    assert np.array_equal(a, draw_num_atoms(data, 1001, seed=3))
    assert not np.array_equal(a, draw_num_atoms(data, 1001, seed=4))
    shards = [a[slice(*shard_range(1001, r, 2))] for r in range(2)]
    assert np.array_equal(np.concatenate(shards), draw_num_atoms(data, 1001, seed=3))
    assert set(a.tolist()) <= set(data.tolist())
    big = draw_num_atoms(data, 100_000, seed=0)
    values, counts = np.unique(data, return_counts=True)
    p = counts / counts.sum()
    freq = np.array([(big == v).mean() for v in values])
    assert np.all(np.abs(freq - p) <= 5 * np.sqrt(p * (1 - p) / 100_000)), (freq, p)


def test_num_atoms_from_refuses_explicit_counts_and_symbols(tmp_path, capsys):
    from arreau_b200 import generate
    base = ["--model_path", str(tmp_path / "missing.ckpt"), "--num_atoms_from", str(tmp_path / "missing.npz")]
    for extra, what in ((["--num_atoms", "8"], "--num_atoms"), (["--symbols", "C", "O"], "--symbols")):
        with pytest.raises(SystemExit):
            generate.main(base + extra)
        assert what in capsys.readouterr().err
    with pytest.raises(ValueError):
        generate.generate_n_crystals(None, 3, None, ["C"], num_atoms=[2, 3, 4])
    with pytest.raises(ValueError):
        generate.generate_n_crystals(None, 3, None, num_atoms=[2, 3])


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _run(device, crystals, **kw):
    from arreau_b200.inference.crystal_metrics import crystal_metrics
    return crystal_metrics(*_pack(crystals), device=device, **kw)


@pytest.mark.gpu
def test_hand_built_cases(device):
    from arreau_b200.inference.crystal_metrics import DEGENERATE, EXTENDED_SEARCH, UNKNOWN_ELEMENT, VALID
    cube5, cube10 = np.eye(3) * 5.0, np.eye(3) * 10.0
    skew = np.array([[4.0, 0, 0], [20.3, 4.0, 0], [0, 0, 4.0]])      # = (4,0,0), (0.3,4,0), (0,0,4) reduced
    skew_f = np.array([[0.0, 0, 0], [0.5, 0.5, 0]])
    cases = [
        ([[0.02, 0.5, 0.5], [0.98, 0.5, 0.5]], cube5, [6, 8]),                 # 0: across a face, 0.2 A
        ([[0, 0, 0], [0.05 + 1e-7, 0, 0]], cube10, [6, 6]),                     # 1: 0.5 A + 1e-6
        ([[0, 0, 0], [0.05 - 1e-7, 0, 0]], cube10, [6, 6]),                     # 2: 0.5 A - 1e-6
        ([[0.3, 0.3, 0.3]], cube5, [26]),                                       # 3: one atom
        ([[0.1, 0.2, 0.3], [0.1, 0.2, 0.3], [0.6, 0.6, 0.6]], cube5, [1, 1, 8]),  # 4: coincident
        ([[0.1, 0.1, 0.1], [0.5, 0.5, 0.5]], np.array([[3.0, 0, 0], [3.0, 0, 0], [0, 0, 3.0]]), [6, 8]),  # 5: V = 0
        ([[0.1, 0.1, 0.1], [0.5, 0.5, 0.5]], np.full((3, 3), np.nan), [6, 8]),  # 6: NaN cell
        ([[0.1, 0.1, 0.1], [0.5, 0.5, 0.5], [0.7, 0.2, 0.9]], cube5, [6, 2001, 6]),  # 7: mask state
        (skew_f, skew, [14, 14]),                                               # 8: 27 images miss the minimum
        ([[0, 0, 0], [0.5, 0, 0]], np.diag([100.0, 1.0, 1.0]), [1, 1]),        # 9: needle beyond the search limit
    ]
    m = _run(device, cases)
    ref = oracle(*_pack(cases[:9]))
    fin = np.isfinite(ref["density"])
    np.testing.assert_allclose(m.volume[:9][fin], ref["volume"][fin], rtol=1e-12, atol=0)
    np.testing.assert_allclose(m.density[:9][fin], ref["density"][fin], rtol=1e-12, atol=0)
    np.testing.assert_allclose(m.min_dist[0], 0.2, rtol=1e-12)
    assert m.flags[0] == 0
    np.testing.assert_allclose(m.min_dist[1:3], [0.5 + 1e-6, 0.5 - 1e-6], rtol=1e-12)
    assert m.flags[1] == VALID and m.flags[2] == 0
    assert m.min_dist[3] == np.inf and m.flags[3] == VALID and m.num_elements[3] == 1
    assert m.min_dist[4] == 0.0 and m.flags[4] == 0 and m.num_elements[4] == 2
    for g in (5, 6):
        assert np.isnan(m.min_dist[g]) and m.flags[g] == DEGENERATE
    assert m.volume[5] == 0.0 and np.isnan(m.volume[6])
    assert m.flags[7] == VALID | UNKNOWN_ELEMENT and np.isnan(m.density[7]) and m.num_elements[7] == 1
    # the 27 images of the given basis miss the nearest image, which the kernel finds
    naive = min(np.linalg.norm((skew_f[1] - skew_f[0] + np.array(k)) @ skew)
                for k in itertools.product((-1, 0, 1), repeat=3))
    true = np.hypot(0.15, 2.0)
    assert naive > true + 2.0
    np.testing.assert_allclose([m.min_dist[8], ref["min_dist"][8]], [true, true], rtol=1e-12)
    assert m.flags[8] & VALID
    # a needle 100 x 1 x 1 with its atoms 50 A apart would need +-51 images across: flagged, not searched
    assert m.flags[9] == DEGENERATE and np.isnan(m.min_dist[9])
    np.testing.assert_array_equal(m.flags[:9] & ~EXTENDED_SEARCH, ref["flags"])


@pytest.mark.gpu
def test_largest_cell_236_atoms(device):
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R
    cr = make_crystals(3, 236, seed=4)
    lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
    z = cr.types + 1
    m = _run(device, [(cr.frac[236 * g:236 * (g + 1)], lat[g], z[236 * g:236 * (g + 1)]) for g in range(3)])
    _assert_matches_oracle(m, oracle(cr.frac, lat, z, cr.num_atoms))


def _synthetic_set(n, seed, sampler_angles=False):
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R
    cr = make_crystals(n, 1, 40, seed=seed)
    angles = cr.angles
    if sampler_angles:     # the sampler's [90, U(90, 180), 90] degrees, consumed as radians
        rng = np.random.default_rng(seed + 1)
        angles = np.stack([np.full(n, 90.0), rng.uniform(90, 180, n), np.full(n, 90.0)], 1)
    lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(angles)).numpy()
    return cr.frac, lat, cr.types + 1, cr.num_atoms


@pytest.mark.gpu
@pytest.mark.parametrize("sampler_angles", [False, True])
def test_random_sets_match_the_oracle(device, sampler_angles):
    from arreau_b200.inference.crystal_metrics import crystal_metrics
    frac, lat, z, na = _synthetic_set(2000, seed=11, sampler_angles=sampler_angles)
    m = crystal_metrics(frac, lat, z, na, device=device)
    _assert_matches_oracle(m, oracle(frac, lat, z, na))
    assert m.valid.any() and (~m.valid).any()
    print(f"extended search: {int(m.extended_search.sum())} of {len(na)}; degenerate {int(m.degenerate.sum())}")


@pytest.mark.gpu
def test_results_do_not_depend_on_batch_or_chunk(device):
    from arreau_b200.inference.crystal_metrics import crystal_metrics
    frac, lat, z, na = _synthetic_set(600, seed=5, sampler_angles=True)
    whole = crystal_metrics(frac, lat, z, na, device=device)
    off = np.concatenate([[0], np.cumsum(na)])
    perm = np.random.default_rng(0).permutation(len(na))
    got = {k: np.empty_like(getattr(whole, k)) for k in ("volume", "min_dist", "density", "num_elements", "flags")}
    for part, chunk_atoms in zip(np.array_split(perm, 3), (1, 97, 1 << 20)):
        idx = np.concatenate([np.arange(off[g], off[g + 1]) for g in part])
        # tensors already on the device for one part, numpy for the others
        args = (frac[idx], lat[part], z[idx], na[part])
        if chunk_atoms == 97:
            args = tuple(torch.as_tensor(a).to(device) for a in args)
        m = crystal_metrics(*args, device=device, max_chunk_atoms=chunk_atoms)
        for k in got:
            got[k][part] = getattr(m, k)
    for k, v in got.items():
        assert v.tobytes() == getattr(whole, k).tobytes(), k


@pytest.mark.gpu
def test_sampler_output_matches_the_oracle(device, weights_npz):
    """A real PONITA_DIFFUSION.sample run (golden weights, T = 11) of 64 crystals with mixed atom counts."""
    from arreau_b200.inference.crystal_metrics import crystal_metrics, sample_inputs
    sys.path.insert(0, os.path.dirname(__file__))
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11)
    counts = np.random.default_rng(2).integers(1, 41, 64)
    np.random.seed(0)
    torch.manual_seed(0)
    res = m.sample(num_atoms_per_sample=None, num_samples_in_batch=64, num_atoms=torch.as_tensor(counts),
                   device=device, device_noise=True, seed=7)
    inputs = sample_inputs(res)
    assert np.array_equal(inputs[3], counts)
    got = crystal_metrics(*inputs, device=device)
    _assert_matches_oracle(got, oracle(*inputs))
    print(f"sampler: {int(got.valid.sum())} valid, {int(got.extended_search.sum())} extended search, "
          f"{int(got.degenerate.sum())} degenerate of 64")


@pytest.mark.gpu
def test_cli_round_trip(device, weights_npz, tmp_path):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    from arreau_b200.generate import draw_num_atoms
    from arreau_b200.inference.crystal_metrics import crystal_metrics, dataset_inputs, sample_inputs, summarize
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R
    sys.path.insert(0, os.path.dirname(__file__))
    from test_gpu_wrapper import _model
    cr = make_crystals(30, 2, 12, seed=21)
    off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
    lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
    data = save_dataset_npz(str(tmp_path / "data"), [cr.types[off[i]:off[i + 1]] % 20 + 1 for i in range(30)], lat,
                            [cr.frac[off[i]:off[i + 1]] for i in range(30)])
    ckpt = str(tmp_path / "model.ckpt")
    _model(device, weights_npz, T=11).save_checkpoint(ckpt)
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = str(tmp_path / "crystals.npz")

    def cli(*args):
        r = subprocess.run([sys.executable, "-m", *args], cwd=ROOT, env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        return r.stdout

    cli("arreau_b200.generate", "--model_path", ckpt, "--num_crystals", "24", "--num_atoms_from", data, "--batch", "10",
        "--precision", "fp32", "--seed", "5", "--out", out)
    js = str(tmp_path / "metrics.json")
    cli("arreau_b200.inference.crystal_metrics", out, "--reference", data, "--json", js)
    inputs = sample_inputs(out)
    assert np.array_equal(inputs[3], draw_num_atoms(cr.num_atoms, 24, seed=5))
    expect = summarize(crystal_metrics(*inputs, device=device),
                       crystal_metrics(*dataset_inputs(CrystalDataset([data])), device=device))
    with open(js) as f:
        assert json.load(f) == json.loads(json.dumps(expect))
    assert expect["reference_frac_valid"] is not None and expect["w1_num_atoms"] is not None
