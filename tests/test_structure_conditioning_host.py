"""Host side of structure-conditioned generation, without a GPU: the checks of known positions, lattices and sites,
the site / composition agreement, known_structures (the --free_elements reordering), the generate CLI's
--structures_from options and its source_index output, and the argument checks of the three known-row entry points."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

Z = 90
NAN = float("nan")


def _loss():
    from arreau_b200.diffusion.diffusion_loss import DiffusionLoss
    return DiffusionLoss(types.SimpleNamespace(radius=5.0, max_neighbors=8, num_timesteps=11), Z)


def _no_engine(monkeypatch, dl):
    def no_engine(*a, **k):
        raise AssertionError("device work before the checks")
    monkeypatch.setattr(dl, "engine_for", no_engine)


def _wrapper(dl):
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    m = PONITA_DIFFUSION.__new__(PONITA_DIFFUSION)
    torch.nn.Module.__init__(m)
    m.register_buffer("z_table_zs", torch.tensor(list(range(1, Z)) + [2001]))
    m.diffusion_loss = dl
    m.t_emb = None
    return m


def test_known_rows_and_lattices():
    from arreau_b200.engine import known_lattices, known_rows
    f = torch.tensor([[0.5, 1.5, -0.25], [NAN, NAN, NAN]])
    v, known = known_rows(f, (2, 3), "known frac")
    assert known.tolist() == [True, False] and v.dtype == torch.float64
    with pytest.raises(ValueError, match="shape"):
        known_rows(f, (3, 3), "known frac")
    with pytest.raises(ValueError, match="row 1 is only partly NaN"):
        known_rows(torch.tensor([[0.5, 0.5, 0.5], [NAN, 0.1, NAN]]), (2, 3), "known frac")
    with pytest.raises(ValueError, match="infinite"):
        known_rows(torch.tensor([[0.5, float("inf"), 0.5]]), (1, 3), "known frac")
    lat = np.stack([np.eye(3) * 4, np.full((3, 3), np.nan), np.diag([1.0, 1.0, 0.05])])
    with pytest.raises(ValueError, match=r"known lattice 2 has \|det\| < 0.1"):
        known_lattices(lat, 3)
    lat[2] = np.diag([1.0, 1.0, 0.11])
    assert known_lattices(lat, 3)[1].tolist() == [True, False, True]
    with pytest.raises(ValueError, match="partly NaN"):
        lat[1, 0, 0] = 1.0
        known_lattices(lat, 3)


def test_sample_refuses_bad_known_parts_before_device_work(monkeypatch):
    dl = _loss()
    _no_engine(monkeypatch, dl)
    kw = dict(model=None, z_table=list(range(Z)), t_emb_weights=None, num_atoms_per_sample=2, num_samples_in_batch=2)
    typed = torch.tensor([3, Z - 1, 5, Z - 1])
    good = torch.tensor([[0.1, 0.2, 0.3], [NAN] * 3, [0.4, 0.5, 0.6], [NAN] * 3])
    with pytest.raises(ValueError, match=r"shape \[4, 3\]"):
        dl.sample(**kw, known_frac=good[:3], initial_types=typed)
    with pytest.raises(ValueError, match="partly NaN"):
        dl.sample(**kw, known_frac=torch.tensor([[0.1, NAN, 0.3]] + [[NAN] * 3] * 3), initial_types=typed)
    with pytest.raises(ValueError, match="infinite"):
        dl.sample(**kw, known_frac=torch.tensor([[0.1, float("-inf"), 0.3]] + [[NAN] * 3] * 3), initial_types=typed)
    with pytest.raises(ValueError, match="known atom 0 has no type"):
        dl.sample(**kw, known_frac=good)                 # every atom starts masked
    with pytest.raises(ValueError, match="known atom 2 has no type"):
        dl.sample(**kw, known_frac=good, initial_types=torch.tensor([3, Z - 1, Z - 1, 1]))
    with pytest.raises(ValueError, match=r"\|det\|"):
        dl.sample(**kw, known_lattice=np.stack([np.eye(3) * 4, np.zeros((3, 3))]))
    with pytest.raises(ValueError, match="shape"):
        dl.sample(**kw, known_lattice=np.stack([np.eye(3)] * 3))
    with pytest.raises(ValueError, match="initial_types must hold 4 states"):
        dl.sample(**kw, initial_types=torch.tensor([3, Z, 5, 1]))
    with pytest.raises(ValueError, match="exclude each other"):
        dl.sample(**kw, initial_types=typed, constant_atoms=typed)
    # constant atoms (compositions) type the known atoms
    with pytest.raises(AssertionError, match="device work"):
        dl.sample(**kw, known_frac=good, constant_atoms=torch.tensor([3, 4, 5, 6]))


def test_wrapper_builds_and_checks_sites_and_lattices(monkeypatch):
    dl = _loss()
    seen = {}

    def fake_sample(**kw):
        seen.clear()
        seen.update(kw)
        return "sampled"
    monkeypatch.setattr(dl, "sample", fake_sample)
    m = _wrapper(dl)
    sites = [(np.array([8, 26]), np.array([[0.1, 0.2, 0.3], [1.25, -0.5, 0.0]])), None, (np.array([], dtype=np.int64),
                                                                                         np.zeros((0, 3)))]
    lat = np.eye(3) * 5
    assert m.sample(3, 3, sites=sites, lattices=[lat, None, lat]) == "sampled"
    kf, it, kl = seen["known_frac"], seen["initial_types"], seen["known_lattice"]
    assert kf.shape == (9, 3) and torch.equal(kf[:2], torch.from_numpy(sites[0][1])) and bool(kf[2:].isnan().all())
    assert it.tolist() == [7, 25] + [Z - 1] * 7                  # sites' states, the rest masked
    assert kl.shape == (3, 3, 3) and np.isnan(kl[1]).all() and np.array_equal(kl[0], lat)
    # compositions type the sites; the first k atomic numbers must agree
    comps = [[8, 26, 3], [3], [1, 1]]
    m.sample(None, 3, compositions=comps, sites=sites)
    assert seen["num_atoms"].tolist() == [3, 1, 2] and "initial_types" not in seen
    assert seen["constant_atoms"].tolist() == [7, 25, 2, 2, 0, 0]
    with pytest.raises(ValueError, match="crystal 0: its composition must begin with its 2 sites"):
        m.sample(None, 3, compositions=[[26, 8, 3], [3], [1, 1]], sites=sites)
    with pytest.raises(ValueError, match="crystal 0 has 2 sites but only 1 atoms"):
        m.sample(1, 3, sites=sites)
    with pytest.raises(ValueError, match=r"\[104\]"):
        m.sample(3, 1, sites=[(np.array([104]), np.zeros((1, 3)))])
    with pytest.raises(ValueError, match="use_constant_atomic_symbols"):
        m.sample(2, 3, sites=sites, use_constant_atomic_symbols=["O", "Fe"])
    with pytest.raises(ValueError, match="sites must hold 3 entries"):
        m.sample(3, 3, sites=sites[:2])
    with pytest.raises(ValueError, match="finite"):
        m.sample(3, 1, sites=[(np.array([8]), np.array([[0.1, NAN, 0.2]]))])
    with pytest.raises(ValueError, match="lattices must hold 3 entries"):
        m.sample(3, 3, lattices=[lat])
    with pytest.raises(ValueError, match="lattice of crystal 1"):
        m.sample(3, 3, lattices=[lat, np.eye(2), None])


def test_generate_refuses_wrong_lengths():
    from arreau_b200.generate import generate_n_crystals
    with pytest.raises(ValueError, match="lattices must hold 3 crystals, got 2"):
        generate_n_crystals(None, 3, 2, lattices=[None, None])
    with pytest.raises(ValueError, match="sites must hold 3 crystals, got 4"):
        generate_n_crystals(None, 3, 2, sites=[None] * 4)


def _dataset(tmp_path, n=30, seed=0):
    from arreau_b200.diffusion.lattice_dataset import save_dataset_npz
    rng = np.random.default_rng(seed)
    zs = [rng.choice([3, 8, 26, 15], rng.integers(1, 9)) for _ in range(n)]
    frac = [rng.random((z.size, 3)) for z in zs]
    lat = np.stack([np.diag(rng.uniform(3, 6, 3)) for _ in range(n)])
    return save_dataset_npz(str(tmp_path / "data.npz"), zs, lat, frac), zs, frac, lat


def test_known_structures_reorders_compositions(tmp_path):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset
    from arreau_b200.generate import known_structures
    path, zs, frac, lat = _dataset(tmp_path)
    ds = CrystalDataset([path])
    idx = np.array([4, 4, 0, 7])
    comps, lats, sites = known_structures(ds, idx, True, ["Li"])
    for i, c, L, s in zip(idx, comps, lats, sites):
        li = zs[i] == 3
        assert np.array_equal(c, np.concatenate([zs[i][~li], zs[i][li]]))   # sites first, then the free atoms
        assert np.array_equal(L, lat[i])
        if li.all():
            assert s is None
        else:
            assert np.array_equal(s[0], zs[i][~li]) and np.array_equal(s[1], frac[i][~li])
    comps, lats, sites = known_structures(ds, idx, True, None)
    assert sites is None and all(np.array_equal(c, zs[i]) for c, i in zip(comps, idx))
    comps, lats, sites = known_structures(ds, idx, False, ["Li", "O"])
    assert lats is None and len(sites) == 4
    with pytest.raises(ValueError, match=r"\['Qq'\]"):
        known_structures(ds, idx, True, ["Li", "Qq"])


def test_generate_cli_structures_from(tmp_path, monkeypatch):
    from test_constrained_host import _fake_cli
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset
    from arreau_b200.generate import draw_compositions, known_structures
    gen, calls = _fake_cli(monkeypatch)
    path, zs, frac, lat = _dataset(tmp_path)
    base = ["--model_path", str(tmp_path / "m.ckpt"), "--num_crystals", "12", "--seed", "5"]
    out = str(tmp_path / "a.npz")
    gen.main(base + ["--structures_from", path, "--fix_lattice", "--free_elements", "Li", "--out", out])
    idx, _ = draw_compositions(CrystalDataset([path]), 12, 5)
    comps, lats, sites = known_structures(CrystalDataset([path]), idx, True, ["Li"])
    c = calls[-1]
    assert all(np.array_equal(a, b) for a, b in zip(c["compositions"], comps))
    assert all(np.array_equal(a, b) for a, b in zip(c["lattices"], lats))
    assert all((a is None and b is None) or (np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]))
               for a, b in zip(c["sites"], sites))
    assert c["elements"] is None and c["num_atoms"] is None
    saved = np.load(out)
    assert np.array_equal(saved["crystals/source_index"], idx)           # seeded: the same draw as draw_compositions
    gen.main(base + ["--structures_from", path, "--fix_lattice", "--out", out])
    assert calls[-1]["sites"] is None and len(calls[-1]["lattices"]) == 12
    gen.main(base + ["--structures_from", path, "--free_elements", "O", "--out", out])
    assert calls[-1]["lattices"] is None and len(calls[-1]["sites"]) == 12
    gen.main(base[:-1] + ["6", "--structures_from", path, "--fix_lattice", "--out", out])
    assert not np.array_equal(np.load(out)["crystals/source_index"], idx)   # another seed, another draw
    n = len(calls)
    refused = [["--structures_from", path], ["--fix_lattice"], ["--free_elements", "Li"],
               ["--structures_from", path, "--fix_lattice", "--free_elements", "Qq"]]
    for extra in (["--num_atoms", "4"], ["--num_atoms_from", path], ["--symbols", "Li"], ["--elements", "Li"],
                  ["--compositions_from", path]):
        refused.append(["--structures_from", path, "--fix_lattice"] + extra)
    for extra in refused:
        with pytest.raises(SystemExit):
            gen.main(base + extra)
    assert len(calls) == n


def test_known_entry_point_argument_checks():
    """Same checks and codes as the entry points without the suffix, plus NULL known buffers; no launch needed."""
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p)
    ve = lambda n, known, x0, fr=p: lib.arreau_ve_pbc_reverse_known(fr, p, p, None, 5, p, n, known, x0, p, None)  # noqa: E731
    assert ve(4, None, p) == -4 and ve(4, p, None) == -4 and ve(4, p, p, fr=None) == -4   # ARREAU_ERR_NULL
    assert ve(-1, p, p) == -1                                                             # ARREAU_ERR_BAD_SHAPE
    assert ve(0, None, None) == 0                                                         # an empty batch is a no-op
    vp = lambda g, t, z, kc, kl, ab: lib.arreau_vp_lattice_reverse_known(  # noqa: E731
        p, p, p, z, t, C.c_double(0.1), C.c_double(0.9), C.c_double(1.0), C.c_double(0.0), g, kc, kl, ab, p, None)
    assert vp(4, 5, p, None, p, p) == -4 and vp(4, 5, p, p, None, p) == -4 and vp(4, 5, p, p, p, None) == -4
    assert vp(4, 5, None, p, p, p) == -4                                                  # z is needed at t > 1
    assert vp(-1, 5, p, p, p, p) == -1
    assert vp(0, 5, None, None, None, None) == 0
    d3 = lambda n, z, coa, allowed, known: lib.arreau_d3pm_reverse_known(  # noqa: E731
        p, p, p, None, 5, p, p, C.c_double(0.98), C.c_double(0.02), 1000, n, z, coa, allowed, known, p, None)
    assert d3(4, 90, None, None, None) == -4           # known_atom is required
    assert d3(4, 90, None, p, p) == -4                 # an allowed set needs crystal_of_atom
    assert d3(4, 500, None, None, p) == -1 and d3(4, 1, None, None, p) == -1 and d3(-1, 90, None, None, p) == -1
    assert d3(0, 90, None, None, None) == 0
    with pytest.raises(RuntimeError, match="ARREAU_ERR_NULL"):
        _lib.call("arreau_ve_pbc_reverse_known", p, p, p, None, 5, p, 4, None, p, p, None)
