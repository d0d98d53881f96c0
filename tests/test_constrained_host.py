"""Host side of chemistry-conditioned generation, without a GPU: the checks of element systems, allowed-state masks and
compositions, draw_compositions, the generate CLI's options and its source_index output, system_fractions, and the
argument checks of arreau_d3pm_reverse_allowed."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

Z = 90


def _z_table():
    from arreau_b200.tools.atomic_number_table import AtomicNumberTable
    return AtomicNumberTable(list(range(1, Z)) + [2001])


def test_element_systems_and_masks():
    from arreau_b200.engine import allowed_state_words
    from arreau_b200.tools.atomic_number_table import allowed_states_of_elements, atomic_numbers_to_states
    zt = _z_table()
    one = allowed_states_of_elements(zt, ["Li", "O", "Li"], 4)
    assert one.shape == (Z,) and np.flatnonzero(one).tolist() == [2, 7]
    per = allowed_states_of_elements(zt, [["H"], ("Fe", "O")], 2)
    assert [np.flatnonzero(r).tolist() for r in per] == [[0], [7, 25]]
    assert not per[:, Z - 1].any()                                  # the mask state is never allowed
    with pytest.raises(ValueError, match="'Xx'"):
        allowed_states_of_elements(zt, ["Li", "Xx"], 1)
    with pytest.raises(ValueError, match="'Lr'"):                   # an element outside the model's z_table
        allowed_states_of_elements(zt, ["Lr"], 1)
    with pytest.raises(ValueError, match="empty"):
        allowed_states_of_elements(zt, [], 1)
    with pytest.raises(ValueError, match="empty"):
        allowed_states_of_elements(zt, [["H"], []], 2)
    with pytest.raises(ValueError, match="3 chemical systems for 2"):
        allowed_states_of_elements(zt, [["H"], ["O"], ["C"]], 2)
    assert atomic_numbers_to_states(zt, [1, 26, 8]).tolist() == [0, 25, 7]
    with pytest.raises(ValueError, match=r"\[104, 2001\]"):
        atomic_numbers_to_states(zt, [1, 2001, 104])
    # packing: bit d of word d // 32; [Z] broadcasts
    w = allowed_state_words(per, 2, Z)
    assert w.dtype == np.uint32 and w.tolist() == [[1, 0, 0, 0], [(1 << 7) | (1 << 25), 0, 0, 0]]
    top = np.zeros(Z, dtype=np.bool_)
    top[[0, 33, 88, Z - 1]] = True
    assert allowed_state_words(top, 3, Z).tolist() == [[1, 2, 1 << 24 | 1 << 25, 0]] * 3
    with pytest.raises(ValueError, match="shape"):
        allowed_state_words(np.ones((2, Z - 1), dtype=np.bool_), 2, Z)
    with pytest.raises(ValueError, match="shape"):
        allowed_state_words(np.ones((3, Z), dtype=np.bool_), 2, Z)
    with pytest.raises(ValueError, match="bool"):
        allowed_state_words(np.ones(Z), 2, Z)
    only_mask = np.zeros((2, Z), dtype=np.bool_)
    only_mask[:, Z - 1] = True
    only_mask[0, 5] = True
    with pytest.raises(ValueError, match="crystal 1 allows no element"):
        allowed_state_words(torch.as_tensor(only_mask), 2, Z)


def test_sample_refuses_bad_options_before_device_work(monkeypatch):
    """DiffusionLoss.sample and PONITA_DIFFUSION.sample raise before any engine is built (none is on this machine)."""
    from arreau_b200.diffusion.diffusion_loss import DiffusionLoss
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    dl = DiffusionLoss(types.SimpleNamespace(radius=5.0, max_neighbors=8, num_timesteps=11), Z)

    def no_engine(*a, **k):
        raise AssertionError("device work before the checks")
    monkeypatch.setattr(dl, "engine_for", no_engine)
    kw = dict(model=None, z_table=list(range(Z)), t_emb_weights=None, num_atoms_per_sample=3, num_samples_in_batch=2)
    with pytest.raises(ValueError, match="shape"):
        dl.sample(**kw, allowed_states=np.ones((3, Z), dtype=np.bool_))
    with pytest.raises(ValueError, match="allows no element"):
        dl.sample(**kw, allowed_states=np.zeros(Z, dtype=np.bool_))
    with pytest.raises(ValueError, match="constant_atoms"):
        dl.sample(**kw, allowed_states=np.ones(Z, dtype=np.bool_), constant_atoms=torch.zeros(6, dtype=torch.int64))
    m = PONITA_DIFFUSION.__new__(PONITA_DIFFUSION)
    torch.nn.Module.__init__(m)
    m.register_buffer("z_table_zs", torch.tensor(list(range(1, Z)) + [2001]))
    m.diffusion_loss = dl
    m.t_emb = None
    with pytest.raises(ValueError, match="'Q'"):
        m.sample(3, 2, elements=["Li", "Q"])
    with pytest.raises(ValueError, match="exclude each other"):
        m.sample(3, 2, elements=["Li"], use_constant_atomic_symbols=["Li"] * 3)
    with pytest.raises(ValueError, match="exclude each other"):
        m.sample(3, 2, elements=["Li"], compositions=[[3], [3]])
    with pytest.raises(ValueError, match="2 non-empty"):
        m.sample(None, 2, compositions=[[3], []])
    with pytest.raises(ValueError, match=r"\[2001\]"):
        m.sample(None, 2, compositions=[[3], [2001]])
    with pytest.raises(ValueError, match="num_atoms"):
        m.sample(None, 2, compositions=[[3], [8]], num_atoms=torch.tensor([1, 1]))


def test_generate_refuses_conflicting_options():
    from arreau_b200.generate import generate_n_crystals
    comps = [np.array([3, 8])] * 3
    for kw in (dict(num_atoms=[2, 2, 2]), dict(use_constant_atomic_symbols=["Li", "O"]), dict(elements=["Li"])):
        with pytest.raises(ValueError, match="compositions"):
            generate_n_crystals(None, 3, None, compositions=comps, **kw)
    with pytest.raises(ValueError, match="3 crystals, got 2"):
        generate_n_crystals(None, 3, None, compositions=comps[:2])
    with pytest.raises(ValueError, match="elements"):
        generate_n_crystals(None, 3, 2, ["Li", "O"], elements=["Li"])
    with pytest.raises(ValueError, match="3 systems, got 2"):
        generate_n_crystals(None, 3, 2, elements=[["Li"], ["O"]])


def _dataset(tmp_path, n=30, seed=0):
    from arreau_b200.diffusion.lattice_dataset import save_dataset_npz
    rng = np.random.default_rng(seed)
    zs = [rng.integers(1, 90, rng.integers(1, 9)) for _ in range(n)]
    frac = [rng.random((z.size, 3)) for z in zs]
    return save_dataset_npz(str(tmp_path / "data.npz"), zs, np.tile(np.eye(3) * 4, (n, 1, 1)), frac), zs


def test_draw_compositions(tmp_path):
    """Seeded, with replacement, the dataset's own compositions, independent of the world size (drawn whole before
    sharding: a rank's shard is a slice of the same draw)."""
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset
    from arreau_b200.distributed import shard_range
    from arreau_b200.generate import draw_compositions
    path, zs = _dataset(tmp_path)
    ds = CrystalDataset([path])
    idx, comps = draw_compositions(ds, 100, seed=3)
    idx2, comps2 = draw_compositions(ds, 100, seed=3)
    assert idx.dtype == np.int64 and idx.shape == (100,) and np.array_equal(idx, idx2)
    assert all(np.array_equal(a, b) for a, b in zip(comps, comps2))
    assert all(np.array_equal(c, zs[i]) for i, c in zip(idx, comps))
    assert len(np.unique(idx)) < 100                                 # with replacement
    assert not np.array_equal(draw_compositions(ds, 100, seed=4)[0], idx)
    parts = [idx[slice(*shard_range(100, r, 3))] for r in range(3)]
    assert np.array_equal(np.concatenate(parts), idx)
    with pytest.raises(ValueError, match="no crystals"):
        draw_compositions(CrystalDataset([]), 5)


def _fake_cli(monkeypatch):
    """generate.main with the model load, the device and the sampler replaced: returns the kwargs of every
    generate_n_crystals call."""
    import arreau_b200.generate as gen
    from arreau_b200.diffusion.diffusion_loss import SampleResult
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    calls = []

    def fake_generate(model, num_crystals, num_atoms_per_sample, symbols, batch, **kw):
        calls.append(dict(num_crystals=num_crystals, num_atoms_per_sample=num_atoms_per_sample, symbols=symbols, **kw))
        na = (np.asarray([len(c) for c in kw["compositions"]]) if kw.get("compositions") is not None else
              np.asarray(kw["num_atoms"]) if kw.get("num_atoms") is not None else np.full(num_crystals, num_atoms_per_sample))
        N = int(na.sum())
        return SampleResult(frac_x=np.zeros((N, 3)), atomic_numbers=np.ones(N, dtype=np.int64),
                            lattice=np.zeros((num_crystals, 3, 3)), num_atoms=na,
                            idx_start=np.concatenate([[0], np.cumsum(na)[:-1]]))
    monkeypatch.setattr(gen, "generate_n_crystals", fake_generate)
    monkeypatch.setattr(PONITA_DIFFUSION, "load_from_checkpoint", classmethod(lambda cls, *a, **k: object()))
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    return gen, calls


def test_generate_cli(tmp_path, monkeypatch):
    from arreau_b200.generate import draw_compositions
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset
    gen, calls = _fake_cli(monkeypatch)
    path, _ = _dataset(tmp_path)
    base = ["--model_path", str(tmp_path / "m.ckpt"), "--num_crystals", "12"]
    out = str(tmp_path / "a.npz")
    gen.main(base + ["--elements", "Li", "Fe", "P", "O", "--num_atoms_from", path, "--out", out])
    assert calls[-1]["elements"] == ["Li", "Fe", "P", "O"] and calls[-1]["num_atoms"].shape == (12,)
    gen.main(base + ["--elements", "Li", "O", "--num_atoms", "6", "--out", out])
    assert calls[-1]["elements"] == ["Li", "O"] and calls[-1]["num_atoms_per_sample"] == 6
    assert calls[-1]["compositions"] is None
    assert "crystals/source_index" not in np.load(out).files
    out = str(tmp_path / "b.npz")
    gen.main(base + ["--compositions_from", path, "--seed", "5", "--out", out])
    idx, comps = draw_compositions(CrystalDataset([path]), 12, 5)
    got = calls[-1]["compositions"]
    assert calls[-1]["elements"] is None and all(np.array_equal(a, b) for a, b in zip(got, comps))
    saved = np.load(out)
    assert np.array_equal(saved["crystals/source_index"], idx)
    assert np.array_equal(saved["crystals/num_atoms"], [c.size for c in comps])
    from arreau_b200.inference.process_generated_crystals import load_sample_results_from_hdf5
    assert load_sample_results_from_hdf5(out).num_atoms.shape == (12,)       # readers of the five keys are unaffected
    n = len(calls)
    for extra in (["--num_atoms", "4"], ["--num_atoms_from", path], ["--symbols", "Li"], ["--elements", "Li"]):
        with pytest.raises(SystemExit):
            gen.main(base + ["--compositions_from", path] + extra)
    with pytest.raises(SystemExit):
        gen.main(base + ["--elements", "Li", "--symbols", "Li", "Li", "Li", "Li"])
    assert len(calls) == n


def test_system_fractions():
    from arreau_b200.inference.crystal_metrics import system_fractions
    z = [3, 26, 15, 8,   3, 3,   3, 26, 15, 8, 1,   8, 15, 26, 3, 3]
    na = [4, 2, 5, 5]
    assert system_fractions(z, na, ["Li", "Fe", "P", "O"]) == dict(frac_in_system=0.75, frac_full_system=0.75)
    assert system_fractions(z, na, ["Li"]) == dict(frac_in_system=0.25, frac_full_system=1.0)
    assert system_fractions(z, na, ["Li", "O", "O"]) == dict(frac_in_system=0.25, frac_full_system=0.75)
    assert system_fractions([], [], ["Li"]) == dict(frac_in_system=None, frac_full_system=None)
    with pytest.raises(ValueError, match="Qq"):
        system_fractions(z, na, ["Li", "Qq"])
    with pytest.raises(ValueError, match="empty"):
        system_fractions(z, na, [])
    with pytest.raises(ValueError, match="does not describe"):
        system_fractions(z, [4, 2], ["Li"])


def test_d3pm_reverse_allowed_argument_checks():
    """Same checks and codes as arreau_d3pm_reverse, plus NULL crystal_of_atom / allowed; no launch needed."""
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p)
    call = lambda n, z, coa, allowed, ty=p: lib.arreau_d3pm_reverse_allowed(  # noqa: E731
        ty, p, p, None, 5, p, p, 0.98, 0.02, 1000, n, z, coa, allowed, p, None)
    assert call(4, 500, p, p) == -1            # Z > 128: ARREAU_ERR_BAD_SHAPE
    assert call(4, 1, p, p) == -1              # Z <= 1
    assert call(-1, 90, p, p) == -1
    assert call(4, 90, None, p) == -4          # ARREAU_ERR_NULL
    assert call(4, 90, p, None) == -4
    assert call(4, 90, p, p, ty=None) == -4
    assert call(0, 90, None, None) == 0        # an empty batch is a no-op
    with pytest.raises(RuntimeError, match="ARREAU_ERR_BAD_SHAPE"):
        _lib.call("arreau_d3pm_reverse_allowed", p, p, p, None, 5, p, p, 0.98, 0.02, 1000, 4, 129, p, p, p, None)
