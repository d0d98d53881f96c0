"""Generation conditioned on chemistry on the GPU: the allowed-state D3PM reverse step (arreau_d3pm_reverse_allowed)
against an fp64 torch restatement of its rule, the whole trajectory with a chemical system per crystal (`elements`),
and per-crystal compositions (`compositions`), through DiffusionLoss.sample, PONITA_DIFFUSION.sample and
generate_n_crystals.  Every comparison of types or trajectories is bit for bit."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

pytestmark = pytest.mark.gpu
Z = 90
T = 1000
EPS = 1e-6


def _restated_reverse(types, logits, u, t_atom, allowed, tb):
    """The constrained reverse step, restated in fp64 torch for every atom (allowed: bool [N,Z], the atom's crystal's
    set with the kernel's normalisation applied: no bit below Z means every state).
    1. x0 probabilities: softmax of the logits over A;  2. argmax candidates: A plus the mask state at t >= 2, A alone
    at t == 1;  posterior log(f1 + eps) + log(f2 + eps) (t >= 2) or the logits (t == 1), plus Gumbel noise scaled by
    1 (t >= 2) or fp32 0.2 (t == 1)."""
    mask = Z - 1
    lg = logits.double().masked_fill(~allowed, float("-inf"))
    p = torch.softmax(lg, dim=1)
    out = torch.empty_like(types)
    d = torch.arange(Z)
    for b in range(types.shape[0]):
        t, xt = int(t_atom[b]), int(types[b])
        gumbel = -torch.log(-torch.log(u[b].clamp(EPS, 1.0)))
        if t == 1:
            val = lg[b] + gumbel * float(np.float32(0.2))
            cand = allowed[b]
        else:
            qa, qb = float(tb.q_keep[t - 2]), float(tb.q_to_mask[t - 2])
            if xt != mask:
                hit, f1_hit, f1_miss = d == xt, tb.onestep_keep, 0.0
            else:
                hit, f1_hit, f1_miss = d == mask, 1.0, tb.onestep_to_mask
            f1 = torch.where(hit, torch.tensor(f1_hit, dtype=torch.float64), torch.tensor(f1_miss, dtype=torch.float64))
            f2 = p[b] * qa
            f2[mask] = p[b, :mask].sum() * qb + p[b, mask]
            val = torch.log(f1 + EPS) + torch.log(f2 + EPS) + gumbel
            cand = allowed[b] | (d == mask)
        val = val.masked_fill(~cand, float("-inf"))
        out[b] = int(torch.argmax(val))
    return out


def _words(allowed_bits):
    """[G,Z+] bool (bits past Z allowed) -> [G,4] int32 words of the kernel."""
    G = allowed_bits.shape[0]
    bits = np.zeros((G, 128), dtype=np.bool_)
    bits[:, :allowed_bits.shape[1]] = allowed_bits
    return np.packbits(bits.reshape(G, 4, 32), axis=-1, bitorder="little").view("<u4").reshape(G, 4).view(np.int32)


def _random_sets(G, rng):
    """Per-crystal sets: one element, many elements, with and without the mask bit, only the mask, no bit below Z
    (unconstrained), every bit, and bits past Z (ignored)."""
    sets = np.zeros((G, 128), dtype=np.bool_)
    for g in range(G):
        kind = g % 7
        if kind == 0:
            sets[g, rng.integers(0, Z - 1)] = True
        elif kind in (1, 2):
            sets[g, rng.choice(Z - 1, rng.integers(2, 30), replace=False)] = True
            sets[g, Z - 1] = kind == 2
        elif kind == 3:
            sets[g, Z - 1] = True
        elif kind == 4:
            sets[g, Z:] = rng.random(128 - Z) < 0.5          # nothing below Z
        elif kind == 5:
            sets[g, :Z] = True
        else:
            sets[g, rng.choice(Z, 5, replace=False)] = True
            sets[g, Z:] = True
    return sets


def test_allowed_reverse_matches_restatement(device):
    """t in {999, 500, 2, 1} (one scalar t per launch, and all four per atom through t_of_atom), 140 crystals with the
    set kinds of _random_sets, atoms masked and already unmasked: the kernel's types equal the restatement's.  With
    every bit set the types equal arreau_d3pm_reverse's."""
    from arreau_b200.tables import build_tables
    tb = build_tables(T, Z)
    rng = np.random.default_rng(0)
    G = 140
    counts = rng.integers(1, 9, G)
    N = int(counts.sum())
    coa = torch.from_numpy(np.repeat(np.arange(G), counts).astype(np.int32))
    sets = _random_sets(G, rng)
    words = _words(sets)
    eff = sets[:, :Z].copy()
    eff[~eff.any(axis=1)] = True                        # no bit below Z: unconstrained
    allowed = torch.from_numpy(eff[coa.numpy()])
    types = torch.from_numpy(np.where(rng.random(N) < 0.5, Z - 1, rng.integers(0, Z - 1, N)).astype(np.int64))
    logits = torch.from_numpy((rng.standard_normal((N, Z)) * 3).astype(np.float32))
    u = torch.from_numpy(rng.random((N, Z)))
    every = _words(np.ones((G, Z), dtype=np.bool_))
    for t in (999, 500, 2, 1):
        got = _reverse(device, types, logits, u, t, None, coa, words, tb)
        want = _restated_reverse(types, logits, u, torch.full((N,), t), allowed, tb)
        assert torch.equal(got, want), (t, int((got != want).sum()))
        assert torch.equal(_reverse(device, types, logits, u, t, None, coa, every, tb),
                           _reverse(device, types, logits, u, t, None, coa, None, tb)), t
    t_atom = torch.from_numpy(rng.choice([999, 500, 2, 1], N))
    got = _reverse(device, types, logits, u, 0, t_atom, coa, words, tb)
    assert torch.equal(got, _restated_reverse(types, logits, u, t_atom, allowed, tb))
    # the sets bind: at t = 1 every atom of a crystal with a set of real elements ends in it
    got = _reverse(device, types, logits, u, 1, None, coa, words, tb)
    assert bool(allowed[torch.arange(N), got].all())


def _reverse(device, types, logits, u, t, t_atom, coa, words, tb):
    from arreau_b200 import _lib
    out = torch.full_like(types, -1, device=device)
    dev = lambda x: x.to(device).contiguous()  # noqa: E731
    ty, lg, uu = dev(types), dev(logits), dev(u)
    ta = None if t_atom is None else dev(t_atom.to(torch.int32))
    qk, qm = dev(tb.q_keep.double()), dev(tb.q_to_mask.double())
    s = torch.cuda.current_stream().cuda_stream
    args = (ty.data_ptr(), lg.data_ptr(), uu.data_ptr(), _lib.ptr(ta), t, qk.data_ptr(), qm.data_ptr(), tb.onestep_keep,
            tb.onestep_to_mask, T, types.shape[0], Z)
    if words is None:
        _lib.call("arreau_d3pm_reverse", *args, out.data_ptr(), s)
    else:
        c, w = dev(coa), dev(torch.from_numpy(words))
        _lib.call("arreau_d3pm_reverse_allowed", *args, c.data_ptr(), w.data_ptr(), out.data_ptr(), s)
    return out.cpu()


def _crystals(res):
    from test_gpu_keyed_sampling import _crystals as c
    return c(res)


def _systems(n, seed):
    """n random chemical systems of 1..6 of the model's elements."""
    from arreau_b200.tools.atomic_number_table import _SYMBOLS
    rng = np.random.default_rng(seed)
    return [[_SYMBOLS[i] for i in rng.choice(Z - 1, rng.integers(1, 7), replace=False)] for _ in range(n)]


def _in_systems(res, systems):
    from arreau_b200.tools.atomic_number_table import ATOMIC_NUMBER
    off = np.concatenate([[0], np.cumsum(res.num_atoms)])
    return all(set(res.atomic_numbers[off[g]:off[g + 1]].tolist()) <= {ATOMIC_NUMBER[e] for e in s}
               for g, s in enumerate(systems))


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_all_states_allowed_equals_unconstrained(device, weights_npz, precision):
    """T = 11: a mask with every state allowed gives the unconstrained trajectory bit for bit, keyed with the CUDA graph
    on and off and with per-batch device noise (whose initial state comes from the host generators, seeded alike for
    both runs)."""
    from test_gpu_keyed_sampling import _population
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision=precision)
    ids, counts = _population(40, 7)
    every = np.ones(Z, dtype=np.bool_)

    def run(allowed, **kw):
        np.random.seed(0)
        torch.manual_seed(0)
        return _crystals(m.sample(None, 40, num_atoms=torch.as_tensor(counts), seed=3, device=device,
                                  allowed_states=allowed, **kw))
    for kw in (dict(crystal_ids=torch.as_tensor(ids)), dict(crystal_ids=torch.as_tensor(ids), cuda_graph=True),
               dict(device_noise=True)):
        assert run(None, **kw) == run(every, **kw), kw


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_elements_trajectories(device, weights_npz, precision):
    """T = 11 with a chemical system per crystal: every final atom is an element of its crystal's system; keyed, a
    crystal's trajectory is the same bits in a batch of 300 and in a permuted batch of 17, CUDA graph on and off; one
    system for every crystal binds too."""
    from test_gpu_keyed_sampling import _population
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision=precision)
    ids, counts = _population(300, 8)
    systems = _systems(300, 9)
    sel = np.random.default_rng(10).permutation(300)[:17]
    runs = {}
    for graph in (False, True):
        for name, idx in (("big", np.arange(300)), ("small", sel)):
            res = m.sample(None, len(idx), num_atoms=torch.as_tensor(counts[idx]), crystal_ids=torch.as_tensor(ids[idx]),
                           seed=5, device=device, cuda_graph=graph, elements=[systems[i] for i in idx])
            assert _in_systems(res, [systems[i] for i in idx])
            runs[(graph, name)] = _crystals(res)
    assert runs[(True, "big")] == runs[(False, "big")] and runs[(True, "small")] == runs[(False, "small")]
    for j, g in enumerate(sel):
        assert runs[(False, "small")][j] == runs[(False, "big")][g], g
    # the constraint changes the outcome, and the engine drops it for the next unconstrained call
    free = _crystals(m.sample(None, 300, num_atoms=torch.as_tensor(counts), crystal_ids=torch.as_tensor(ids), seed=5,
                              device=device))
    assert free != runs[(False, "big")]
    one = m.sample(None, 300, num_atoms=torch.as_tensor(counts), crystal_ids=torch.as_tensor(ids), seed=5, device=device,
                   elements=["Li", "Fe", "P", "O"], cuda_graph=True)
    assert _in_systems(one, [["Li", "Fe", "P", "O"]] * 300)
    again = _crystals(m.sample(None, 300, num_atoms=torch.as_tensor(counts), crystal_ids=torch.as_tensor(ids), seed=5,
                               device=device))
    assert again == free


def _world2(rank):
    class World2:       # generate_n_crystals' view of a 2-rank run; the final gather stays local
        def is_initialized(self):
            return True

        def get_rank(self, group=None):
            return rank

        def get_world_size(self, group=None):
            return 2
    return World2()


def test_generate_compositions(device, weights_npz, monkeypatch):
    """Per-crystal compositions: the final types are the input, keyed runs are bit-identical at batch 1000 and 17 and
    over two emulated ranks, and identical compositions give what use_constant_atomic_symbols gives, bit for bit (one
    crystal per batch, where the reference's per-batch np.repeat layout of the symbols is the composition itself; and a
    one-element composition at any batch)."""
    import arreau_b200.generate as gen
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision="fp16")
    rng = np.random.default_rng(11)
    comps = [rng.choice(np.arange(1, Z), rng.integers(1, 25)) for _ in range(41)]
    run = lambda **kw: gen.generate_n_crystals(m, 41, None, device=device, seed=9, keyed_noise=True, **kw)  # noqa: E731
    whole = run(compositions=comps, num_crystals_per_batch=1000)
    assert np.array_equal(whole.atomic_numbers, np.concatenate(comps))
    assert np.array_equal(whole.num_atoms, [c.size for c in comps])
    assert _crystals(run(compositions=comps, num_crystals_per_batch=17)) == _crystals(whole)
    shards = []
    for r in range(2):
        monkeypatch.setattr(gen, "dist", _world2(r))
        shards.append(run(compositions=comps, num_crystals_per_batch=8))
    monkeypatch.undo()
    assert _crystals(shards[0]) + _crystals(shards[1]) == _crystals(whole)
    for symbols, batch in ((["Li", "Fe", "P", "O", "O", "O", "O"], 1), (["Si"] * 5, 6)):
        from arreau_b200.tools.atomic_number_table import ATOMIC_NUMBER
        z = np.asarray([ATOMIC_NUMBER[e] for e in symbols])
        ref = gen.generate_n_crystals(m, 6, len(symbols), symbols, num_crystals_per_batch=batch, device=device, seed=4,
                                      keyed_noise=True)
        got = gen.generate_n_crystals(m, 6, None, compositions=[z] * 6, num_crystals_per_batch=1000, device=device,
                                      seed=4, keyed_noise=True)
        assert _crystals(got) == _crystals(ref), symbols


def test_generate_elements_shards(device, weights_npz, monkeypatch):
    """Per-crystal systems with per-crystal atom counts: two emulated ranks equal the whole run, which equals a run at
    another batch size; every atom is in its crystal's system."""
    import arreau_b200.generate as gen
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision="fp16")
    counts = np.random.default_rng(12).integers(1, 30, 41)
    systems = _systems(41, 13)
    run = lambda **kw: gen.generate_n_crystals(m, 41, None, num_atoms=counts, device=device, seed=9,  # noqa: E731
                                               keyed_noise=True, elements=systems, **kw)
    whole = run(num_crystals_per_batch=1000)
    assert _in_systems(whole, systems)
    assert _crystals(run(num_crystals_per_batch=17)) == _crystals(whole)
    shards = []
    for r in range(2):
        monkeypatch.setattr(gen, "dist", _world2(r))
        shards.append(run(num_crystals_per_batch=8))
    monkeypatch.undo()
    assert _crystals(shards[0]) + _crystals(shards[1]) == _crystals(whole)
