"""Per-crystal keyed sampling noise on the GPU: the draws of arreau_sample_init_keyed / arreau_sample_noise_keyed, whole
sampler trajectories, generate_n_crystals(keyed_noise=True), and sample-quality monitoring inside train.fit.

Every comparison of a crystal across batch layouts, CUDA graph on / off, world sizes, or runs with and without
monitoring is bit for bit (tobytes / torch.equal).  The moment checks allow 6 standard errors."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

pytestmark = pytest.mark.gpu
Z = 90


def _topology(counts, device):
    counts = np.asarray(counts, dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    coa = np.repeat(np.arange(len(counts)), counts).astype(np.int32)
    return torch.from_numpy(off).to(device), torch.from_numpy(coa).to(device)


def _draw(device, ids, counts, seed, steps):
    """(angles, lengths, frac) of the initial state and (z_len, z_frac, u) of every step in `steps`, as host arrays."""
    from arreau_b200 import _lib
    from arreau_b200.tables import POS_SIGMA_MAX
    G, N = len(ids), int(np.sum(counts))
    off, coa = _topology(counts, device)
    cid = torch.as_tensor(np.asarray(ids, dtype=np.int64)).to(device)
    f64 = lambda *s: torch.full(s, float("nan"), dtype=torch.float64, device=device)  # noqa: E731
    angles, lengths, frac = f64(G, 3), f64(G, 3), f64(N, 3)
    s = torch.cuda.current_stream().cuda_stream
    _lib.call("arreau_sample_init_keyed", C.c_uint64(seed), G, N, cid.data_ptr(), off.data_ptr(), coa.data_ptr(),
              POS_SIGMA_MAX, angles.data_ptr(), lengths.data_ptr(), frac.data_ptr(), s)
    out = {"init": [t.cpu().numpy() for t in (angles, lengths, frac)]}
    for k in steps:
        z_len, z_frac, u = f64(G, 3), f64(N, 3), f64(N, Z)
        _lib.call("arreau_sample_noise_keyed", C.c_uint64(seed), k, G, N, Z, cid.data_ptr(), off.data_ptr(),
                  coa.data_ptr(), z_len.data_ptr(), z_frac.data_ptr(), u.data_ptr(), s)
        out[k] = [t.cpu().numpy() for t in (z_len, z_frac, u)]
    return out


def _population(n, seed):
    rng = np.random.default_rng(seed)
    ids = rng.choice(1 << 20, n, replace=False).astype(np.int64) + (np.int64(1) << 40)   # ids that need 64 bits
    counts = rng.integers(1, 41, n)
    return ids, counts


def test_keyed_draws_do_not_depend_on_the_batch(device):
    """A crystal's initial state and step noise are the same bits at any position of batches of 300 and 17 crystals
    with mixed atom counts; the moments are those of the reference's distributions."""
    from arreau_b200 import _lib
    from arreau_b200.tables import POS_SIGMA_MAX
    ids, counts = _population(300, 1)
    steps = [0, 1, 997, (1 << 28) - 1]
    big = _draw(device, ids, counts, 11, steps)
    sel = np.random.default_rng(2).permutation(300)[:17]
    small = _draw(device, ids[sel], counts[sel], 11, steps)
    for key in ["init"] + steps:
        # per-crystal arrays first: [G,3] (angles, lengths / z_len), then per-atom ones
        G = len(ids)
        a_rows = [_split(x, counts, G) for x in big[key]]
        b_rows = [_split(x, counts[sel], len(sel)) for x in small[key]]
        for j, g in enumerate(sel):
            for xa, xb in zip(a_rows, b_rows):
                assert xa[g] == xb[j], (key, g)
    # different steps, different draws; another seed, other draws
    assert not np.array_equal(big[0][1], big[1][1]) and not np.array_equal(big[0][2], big[(1 << 28) - 1][2])
    other = _draw(device, ids, counts, 12, [0])
    assert not np.array_equal(other[0][1], big[0][1]) and not np.array_equal(other["init"][2], big["init"][2])
    # distributions
    angles, lengths, frac = big["init"]
    assert np.all(angles[:, 0] == 90.0) and np.all(angles[:, 2] == 90.0)
    beta = angles[:, 1]
    assert beta.min() >= 90.0 and beta.max() < 180.0
    _assert_uniform((beta - 90.0) / 90.0)
    _assert_normal(lengths.ravel())
    _assert_normal((frac / POS_SIGMA_MAX).ravel())
    for k in steps:
        z_len, z_frac, u = big[k]
        _assert_normal(np.concatenate([z_len.ravel(), z_frac.ravel()]))
        assert u.min() >= 0.0 and u.max() < 1.0
        _assert_uniform(u.ravel())
    # the counter layout bounds the step ordinal
    lib = _lib.load()
    buf = torch.zeros(64, dtype=torch.float64, device=device)
    p = buf.data_ptr()
    assert lib.arreau_sample_noise_keyed(C.c_uint64(0), 1 << 28, 1, 1, Z, p, p, p, p, p, p, None) == -1
    assert lib.arreau_sample_noise_keyed(C.c_uint64(0), -1, 1, 1, Z, p, p, p, p, p, p, None) == -1
    assert lib.arreau_sample_init_keyed(C.c_uint64(0), 1, 1, None, p, p, 1.0, p, p, p, None) == -4


def _split(x, counts, G):
    off = np.concatenate([[0], np.cumsum(counts)])
    if x.shape[0] == G:
        return [x[g].tobytes() for g in range(G)]
    return [x[off[g]:off[g + 1]].tobytes() for g in range(G)]


def _assert_normal(v):
    n = v.size
    assert np.isfinite(v).all()
    assert abs(v.mean()) < 6 / np.sqrt(n), v.mean()
    assert abs(v.var() - 1.0) < 6 * np.sqrt(2.0 / n), v.var()


def _assert_uniform(v):
    n = v.size
    assert abs(v.mean() - 0.5) < 6 * np.sqrt(1 / 12 / n), v.mean()
    assert abs(v.var() - 1 / 12) < 6 * np.sqrt(1 / 180 / n), v.var()


def _rng_states():
    return (torch.get_rng_state().clone(), torch.cuda.get_rng_state().clone(), np.random.get_state())


def _same_rng(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert a[2][0] == b[2][0] and np.array_equal(a[2][1], b[2][1]) and a[2][2:] == b[2][2:]


def _crystals(res):
    """Per crystal (frac bytes, atomic numbers bytes, lattice bytes) of a SampleResult."""
    na = np.asarray(res.num_atoms)
    off = np.concatenate([[0], np.cumsum(na)])
    return [(res.frac_x[off[g]:off[g + 1]].tobytes(), np.asarray(res.atomic_numbers[off[g]:off[g + 1]]).tobytes(),
             res.lattice[g].tobytes()) for g in range(len(na))]


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_keyed_trajectories_do_not_depend_on_the_batch(device, weights_npz, precision):
    """T = 11: a crystal's final frac, types and lattice are the same bits in a batch of 300 and in a batch of 17 in
    another order, with the CUDA graph on and off; a keyed sample leaves the torch and numpy generators as they were."""
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision=precision)
    ids, counts = _population(300, 3)
    sel = np.random.default_rng(4).permutation(300)[:17]
    runs = {}
    before = _rng_states()
    for graph in (False, True):
        for name, idx in (("big", np.arange(300)), ("small", sel)):
            res = m.sample(None, len(idx), num_atoms=torch.as_tensor(counts[idx]), crystal_ids=torch.as_tensor(ids[idx]),
                           seed=5, device=device, cuda_graph=graph)
            assert np.array_equal(res.num_atoms, counts[idx])
            runs[(graph, name)] = _crystals(res)
    _same_rng(before, _rng_states())
    assert runs[(True, "big")] == runs[(False, "big")] and runs[(True, "small")] == runs[(False, "small")]
    big, small = runs[(False, "big")], runs[(False, "small")]
    for j, g in enumerate(sel):
        assert small[j] == big[g], g
    # the state moved off its start, and the noise is per crystal: crystals with equal counts differ
    same = [g for g in range(300) if counts[g] == counts[sel[0]] and g != sel[0]]
    assert same and all(big[g][0] != big[sel[0]][0] for g in same)
    # constant atoms: the types stay, the rest is keyed the same way
    ca = torch.full((int(counts[sel].sum()),), 5, dtype=torch.int64)
    res = m.diffusion_loss.sample(model=m, z_table=list(range(1, Z)) + [2001], t_emb_weights=m.t_emb,
                                  num_atoms_per_sample=None, num_samples_in_batch=17, num_atoms=torch.as_tensor(counts[sel]),
                                  constant_atoms=ca, crystal_ids=torch.as_tensor(ids[sel]), seed=5, device=device)
    assert np.all(res.atomic_numbers == 6)


def test_generate_keyed_noise_does_not_depend_on_batch_or_world(device, weights_npz, monkeypatch):
    import arreau_b200.generate as gen
    from arreau_b200.distributed import shard_range
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision="fp16")
    counts = np.random.default_rng(6).integers(1, 30, 41)
    run = lambda **kw: gen.generate_n_crystals(m, 41, None, num_atoms=counts, device=device, seed=9, **kw)  # noqa: E731
    whole = run(keyed_noise=True, num_crystals_per_batch=1000)
    batched = run(keyed_noise=True, num_crystals_per_batch=17)
    assert _crystals(whole) == _crystals(batched)
    assert np.array_equal(whole.idx_start, batched.idx_start) and np.array_equal(whole.num_atoms, counts)

    class World2:       # generate_n_crystals' view of a 2-rank run; the final gather stays local
        def __init__(self, rank):
            self.rank = rank

        def is_initialized(self):
            return True

        def get_rank(self, group=None):
            return self.rank

        def get_world_size(self, group=None):
            return 2

    shards = []
    for r in range(2):
        monkeypatch.setattr(gen, "dist", World2(r))
        shards.append(run(keyed_noise=True, num_crystals_per_batch=8))
        lo, hi = shard_range(41, r, 2)
        assert np.array_equal(shards[-1].num_atoms, counts[lo:hi])
    monkeypatch.undo()
    assert _crystals(shards[0]) + _crystals(shards[1]) == _crystals(whole)
    # without the option: batch b0 is sampled with seed + b0 and the host generators, as before
    np.random.seed(0)
    torch.manual_seed(0)
    plain = run(num_crystals_per_batch=17)
    np.random.seed(0)
    torch.manual_seed(0)
    expect = []
    for b0 in range(0, 41, 17):
        nb = min(17, 41 - b0)
        expect += _crystals(m.sample(None, nb, num_atoms=torch.as_tensor(counts[b0:b0 + nb]), device=device,
                                     device_noise=True, seed=9 + b0))
    assert _crystals(plain) == expect and _crystals(plain) != _crystals(whole)


def _dataset(tmp_path, n, seed):
    from test_gpu_resume import _dataset as ds
    return ds(tmp_path, n, seed)


def _quiet(*_):
    pass


def _standalone_record(device, ckpt, train, reference, count, seed, epoch):
    """summarize of a keyed generate with a checkpoint's weights plus crystal_metrics, as a quality_record."""
    from arreau_b200.generate import draw_num_atoms, generate_n_crystals
    from arreau_b200.inference.crystal_metrics import (crystal_metrics, dataset_inputs, quality_record, sample_inputs,
                                                       summarize)
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    m = PONITA_DIFFUSION.load_from_checkpoint(str(ckpt), precision="fp16").to(device)
    counts = draw_num_atoms(train.atom_counts(), count, seed)
    res = generate_n_crystals(m, count, None, num_atoms=counts, keyed_noise=True, seed=seed, device=device,
                              num_crystals_per_batch=10)
    ref = crystal_metrics(*dataset_inputs(reference), device=device)
    return quality_record(summarize(crystal_metrics(*sample_inputs(res), device=device), ref), epoch)


@pytest.mark.parametrize("ema", [None, 0.9])
def test_fit_sample_quality(device, tmp_path, ema):
    """fit with sample_every = 2 over 3 epochs (passes after epochs 1 and 2): training is bit-identical to a run without
    monitoring; each record equals a standalone keyed generate + crystal_metrics on that epoch's saved weights; a run
    stopped after epoch 1 and resumed returns the same history bit for bit."""
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION, load_checkpoint_file
    from arreau_b200.train import ema_path, fit
    from test_gpu_resume import _cli_splits, _model
    _, ds = _dataset(tmp_path, 64, seed=5)
    tr, va = _cli_splits(ds, 0.25)
    M = 24
    run = dict(batch_size=12, device=device, val_dataset=va, ema_decay=ema, log=_quiet, seed=0)
    lines = []
    plain = _model(ds, lr=1e-3, epochs=3)
    h_plain = fit(plain, tr, 3, **run)
    mon, met = _model(ds, lr=1e-3, epochs=3), {}
    h_mon = fit(mon, tr, 3, checkpoint_dir=str(tmp_path / "a"), metrics=met, sample_every=2, sample_count=M,
                **{**run, "log": lines.append})
    assert h_mon == h_plain and torch.equal(mon.model.flat.data, plain.model.flat.data)
    assert torch.equal(mon._optimizer.exp_avg, plain._optimizer.exp_avg)
    if ema is not None:
        assert torch.equal(mon._optimizer.ema.data, plain._optimizer.ema.data)
    assert [r["epoch"] for r in met["samples"]] == [1, 2] and met["sample_quality"] == met["samples"]
    assert "samples: valid" in lines[1] and "samples" not in lines[0] and "samples: valid" in lines[2]
    print("sample quality:", met["samples"])
    fs = load_checkpoint_file(str(tmp_path / "a" / "last.ckpt"))["fit_state"]
    assert fs["sample_quality"] == met["samples"] and (fs["sample_every"], fs["sample_count"]) == (2, M)
    # stopped after epoch 1, then resumed in a new model
    first, met_1 = _model(ds, lr=1e-3, epochs=3), {}
    fit(first, tr, 2, checkpoint_dir=str(tmp_path / "b"), metrics=met_1, sample_every=2, sample_count=M, **run)
    assert met_1["samples"] == met["samples"][:1]
    name = "last.ckpt" if ema is None else ema_path("last.ckpt")
    assert met_1["samples"][0] == _standalone_record(device, tmp_path / "b" / name, tr, va, M, 0, 1)
    last = str(tmp_path / "b" / "last.ckpt")
    resumed, met_r = PONITA_DIFFUSION.load_from_checkpoint(last), {}
    fit(resumed, tr, 3, checkpoint_dir=str(tmp_path / "b"), metrics=met_r, resume_from=last, sample_every=2,
        sample_count=M, **run)
    assert met_r["samples"] == met["samples"][1:] and met_r["sample_quality"] == met["samples"]
    assert load_checkpoint_file(last)["fit_state"]["sample_quality"] == met["samples"]
    assert torch.equal(resumed.model.flat.data, mon.model.flat.data)
    assert met["samples"][1] == _standalone_record(device, tmp_path / "a" / name, tr, va, M, 0, 2)
