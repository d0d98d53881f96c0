"""Generation conditioned on structure on the GPU: the known-row reverse steps (arreau_ve_pbc_reverse_known,
arreau_vp_lattice_reverse_known, arreau_d3pm_reverse_known) against the forward kernels at level t-1 and the existing
reverse kernels, and whole trajectories with known lattices and known sites through DiffusionLoss.sample,
PONITA_DIFFUSION.sample and generate_n_crystals.  Every comparison of positions, lengths, types or trajectories is bit
for bit; only the final lattice is compared through its Gram matrix (the cell may be given in any orientation)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

pytestmark = pytest.mark.gpu
Z = 90
T = 1000


def _known_mask(counts, rng):
    """Per atom: known or free.  Crystal g % 3 == 0 is all known, 1 all free, 2 mixed."""
    return np.concatenate([np.ones(n, bool) if g % 3 == 0 else np.zeros(n, bool) if g % 3 == 1 else rng.random(n) < 0.5
                           for g, n in enumerate(counts)])


def _setup(device, seed=0):
    from arreau_b200.tables import build_tables
    rng = np.random.default_rng(seed)
    G = 60
    counts = rng.integers(1, 9, G)
    N = int(counts.sum())
    d = lambda a: torch.as_tensor(a).to(device).contiguous()  # noqa: E731
    s = dict(tb=build_tables(T, Z), G=G, N=N, counts=counts, rng=rng,
             known_atom=_known_mask(counts, rng), known_crystal=np.arange(G) % 3 != 1,
             frac=d(rng.random((N, 3))), score=d(rng.standard_normal((N, 3)).astype(np.float32)),
             z_frac=d(rng.standard_normal((N, 3))), x0=d(rng.random((N, 3))),
             lengths=d(rng.standard_normal((G, 3)) + 5), len0=d(rng.random((G, 3)).astype(np.float32)),
             z_len=d(rng.standard_normal((G, 3))), l0=d(rng.random((G, 3)) * 5 + 2),
             types=d(np.where(rng.random(N) < 0.5, Z - 1, rng.integers(0, Z - 1, N)).astype(np.int64)),
             logits=d((rng.standard_normal((N, Z)) * 3).astype(np.float32)), u=d(rng.random((N, Z))))
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    s.update(atom_offset=d(off), coa=d(np.repeat(np.arange(G), counts).astype(np.int32)),
             ka=d(s["known_atom"].astype(np.int32)), kc=d(s["known_crystal"].astype(np.int32)))
    return s


def _ve(device, s, t, t_atom, known):
    from arreau_b200 import _lib
    out = torch.full_like(s["frac"], -1.0)
    sig = s["tb"].ve_sigmas.to(device)
    ta = None if t_atom is None else t_atom.to(device, torch.int32)
    args = (s["frac"].data_ptr(), s["score"].data_ptr(), s["z_frac"].data_ptr(), _lib.ptr(ta), t, sig.data_ptr(), s["N"])
    stream = torch.cuda.current_stream().cuda_stream
    if known:
        _lib.call("arreau_ve_pbc_reverse_known", *args, s["ka"].data_ptr(), s["x0"].data_ptr(), out.data_ptr(), stream)
    else:
        _lib.call("arreau_ve_pbc_reverse", *args, out.data_ptr(), stream)
    return out.cpu()


def _vp(device, s, t, known):
    from arreau_b200 import _lib
    tb = s["tb"]
    out = torch.full_like(s["lengths"], -1.0)
    ab = tb.vp_alpha_bars.to(device, torch.float32)
    args = (s["lengths"].data_ptr(), s["len0"].data_ptr(), s["atom_offset"].data_ptr(), s["z_len"].data_ptr(), t,
            float(tb.vp_cx0[t]), float(tb.vp_cxt[t]), float(tb.vp_denom[t]), float(tb.vp_var[t]), s["G"])
    stream = torch.cuda.current_stream().cuda_stream
    if known:
        _lib.call("arreau_vp_lattice_reverse_known", *args, s["kc"].data_ptr(), s["l0"].data_ptr(), ab.data_ptr(),
                  out.data_ptr(), stream)
    else:
        _lib.call("arreau_vp_lattice_reverse", *args, out.data_ptr(), stream)
    return out.cpu()


def _d3pm(device, s, t, t_atom, known, words):
    from arreau_b200 import _lib
    tb = s["tb"]
    out = torch.full_like(s["types"], -1)
    ta = None if t_atom is None else t_atom.to(device, torch.int32)
    qk, qm = tb.q_keep.double().to(device), tb.q_to_mask.double().to(device)
    w = None if words is None else torch.from_numpy(words).to(device)
    args = (s["types"].data_ptr(), s["logits"].data_ptr(), s["u"].data_ptr(), _lib.ptr(ta), t, qk.data_ptr(),
            qm.data_ptr(), tb.onestep_keep, tb.onestep_to_mask, T, s["N"], Z)
    stream = torch.cuda.current_stream().cuda_stream
    if known:
        _lib.call("arreau_d3pm_reverse_known", *args, s["coa"].data_ptr(), _lib.ptr(w), s["ka"].data_ptr(),
                  out.data_ptr(), stream)
    elif w is not None:
        _lib.call("arreau_d3pm_reverse_allowed", *args, s["coa"].data_ptr(), w.data_ptr(), out.data_ptr(), stream)
    else:
        _lib.call("arreau_d3pm_reverse", *args, out.data_ptr(), stream)
    return out.cpu()


def test_known_reverse_steps_match_forward_oracle(device):
    """t in {999, 500, 2, 1} (scalar t, and the four mixed per atom through t_of_atom): a known row equals the forward
    kernel at level t-1 with the row's own step noise (t >= 2), or x0 / l0 exactly (t == 1); a free row equals the
    existing reverse kernel; a known atom keeps its type, with and without an allowed-state set."""
    from arreau_b200.diffusion.diffusion_helpers import VE_pbc, VP_lattice
    from arreau_b200.tables import POS_SIGMA_MAX, POS_SIGMA_MIN
    from test_gpu_constrained_sampling import _random_sets, _words
    s = _setup(device)
    G, N = s["G"], s["N"]
    ka, kc = torch.from_numpy(s["known_atom"]), torch.from_numpy(s["known_crystal"])
    ve, vp = VE_pbc(T, POS_SIGMA_MIN, POS_SIGMA_MAX), VP_lattice(T)
    assert torch.equal(ve.sigmas, s["tb"].ve_sigmas)
    lattice = torch.eye(3, dtype=torch.float64, device=device).repeat(G, 1, 1) * 4
    na = torch.as_tensor(s["counts"])
    words = _words(_random_sets(G, s["rng"]))
    x0, l0 = s["x0"].cpu(), s["l0"].cpu()

    def ve_oracle(t_atom):          # forward at level t-1 for t >= 2, x0 at t == 1
        fwd = ve.forward(s["x0"], (t_atom - 1).clamp_min(0).to(device), lattice, na, noise=s["z_frac"])[0].cpu()
        return torch.where((t_atom == 1)[:, None], x0, fwd)

    for t in (999, 500, 2, 1):
        t_atom = torch.full((N,), t)
        got, free = _ve(device, s, t, None, True), _ve(device, s, t, None, False)
        assert torch.equal(got[ka], ve_oracle(t_atom)[ka]), t
        assert torch.equal(got[~ka], free[~ka]), t
        if t == 1:
            assert torch.equal(got[ka], x0[ka])
        got, free = _vp(device, s, t, True), _vp(device, s, t, False)
        want = vp.forward(s["l0"], torch.full((G,), max(t - 1, 0), device=device), noise=s["z_len"])[0].cpu()
        assert torch.equal(got[kc], (want if t >= 2 else l0)[kc]), t
        assert torch.equal(got[~kc], free[~kc]), t
        if t == 1:
            assert torch.equal(got[kc], l0[kc])
        for w in (None, words):
            got, free = _d3pm(device, s, t, None, True, w), _d3pm(device, s, t, None, False, w)
            assert torch.equal(got[ka], s["types"].cpu()[ka]), t
            assert torch.equal(got[~ka], free[~ka]), t
    t_atom = torch.from_numpy(s["rng"].choice([999, 500, 2, 1], N))
    got, free = _ve(device, s, 0, t_atom, True), _ve(device, s, 0, t_atom, False)
    assert torch.equal(got[ka], ve_oracle(t_atom)[ka])
    assert torch.equal(got[~ka], free[~ka])
    for w in (None, words):
        got, free = _d3pm(device, s, 0, t_atom, True, w), _d3pm(device, s, 0, t_atom, False, w)
        assert torch.equal(got[ka], s["types"].cpu()[ka]) and torch.equal(got[~ka], free[~ka])
    # nothing known: the known instances give the existing kernels' output on every row
    s["ka"].zero_()
    s["kc"].zero_()
    assert torch.equal(_ve(device, s, 500, None, True), _ve(device, s, 500, None, False))
    assert torch.equal(_vp(device, s, 500, True), _vp(device, s, 500, False))
    assert torch.equal(_d3pm(device, s, 1, None, True, None), _d3pm(device, s, 1, None, False, None))


def _crystals(res):
    from test_gpu_keyed_sampling import _crystals as c
    return c(res)


def _wrap(x):
    """Known positions as the engine stores them: torch.remainder(x, 1), with the 1.0 it gives for tiny negative x
    mapped to 0.0."""
    w = torch.remainder(torch.from_numpy(x), 1.0)
    return torch.where(w == 1.0, torch.zeros_like(w), w).numpy()


def _lattices(G, rng, every=3):
    """A random cell (lengths 3..7 A, skewed) for every crystal but each `every`-th, which is None."""
    return [None if g % every == 1 else np.diag(rng.uniform(3, 7, 3)) + rng.uniform(-1, 1, (3, 3)) for g in range(G)]


def _sites(counts, rng, comps=None):
    """Per crystal: None, all atoms, or its first k of n atoms (k random) as sites, at positions partly outside [0,1)
    (they are wrapped).  With `comps` the sites' atomic numbers are the composition's first k."""
    out = []
    for g, n in enumerate(counts):
        kind = g % 3
        if kind == 1:
            out.append(None)
            continue
        k = int(n) if kind == 0 else int(rng.integers(0, n + 1))
        z = comps[g][:k] if comps is not None else rng.integers(1, Z, k)
        out.append((np.asarray(z), rng.uniform(-0.5, 1.5, (k, 3))))
    return out


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_nothing_known_equals_unconditioned(device, weights_npz, precision):
    """T = 11: all-NaN known buffers (the conditioned kernels run, no row is known) give the unconditioned trajectory
    bit for bit, keyed and with per-batch device noise (whose initial state comes from the host generators, seeded
    alike for both runs), each with the CUDA graph on and off."""
    from test_gpu_keyed_sampling import _population
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision=precision)
    ids, counts = _population(40, 7)
    N = int(counts.sum())
    empty = dict(known_frac=torch.full((N, 3), float("nan")), known_lattice=torch.full((40, 3, 3), float("nan")))

    def run(known, **kw):
        np.random.seed(0)
        torch.manual_seed(0)
        return _crystals(m.sample(None, 40, num_atoms=torch.as_tensor(counts), seed=3, device=device,
                                  **(empty if known else {}), **kw))
    for kw in (dict(crystal_ids=torch.as_tensor(ids)), dict(crystal_ids=torch.as_tensor(ids), cuda_graph=True),
               dict(device_noise=True), dict(device_noise=True, cuda_graph=True)):
        assert run(False, **kw) == run(True, **kw), kw


@pytest.mark.parametrize("graph", [False, True])
def test_final_state_holds_the_known_structure(device, weights_npz, graph):
    """T = 11, keyed: known atoms end exactly at their wrapped positions with their elements, known-lattice crystals
    end with exactly the known lengths and a lattice with the given Gram matrix; the free atoms differ from an
    unconditioned run's (the conditioning reaches the model)."""
    from arreau_b200.diffusion.lattice_helpers import matrix_to_params
    from test_gpu_keyed_sampling import _population
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision="fp16")
    G = 60
    ids, counts = _population(G, 21)
    rng = np.random.default_rng(22)
    lats, sites = _lattices(G, rng), _sites(counts, rng)
    sites[0][1][0, 0] = -1e-20                 # wraps to 1.0 under remainder; stored as 0.0
    kw = dict(num_atoms=torch.as_tensor(counts), crystal_ids=torch.as_tensor(ids), seed=4, device=device,
              cuda_graph=graph)
    res = m.sample(None, G, lattices=lats, sites=sites, **kw)
    lengths = m.diffusion_loss._engine.lengths.cpu()
    free_run = m.sample(None, G, **kw)
    off = np.concatenate([[0], np.cumsum(counts)])
    free_rows = np.ones(off[-1], bool)
    for g in range(G):
        if sites[g] is not None:
            z, x = sites[g]
            k = z.shape[0]
            rows = slice(off[g], off[g] + k)
            assert res.frac_x[rows].tobytes() == _wrap(x).tobytes(), g
            assert np.array_equal(res.atomic_numbers[rows], z), g
            free_rows[rows] = False
        if lats[g] is not None:
            L = torch.from_numpy(lats[g][None]).to(device)
            assert torch.equal(lengths[g], matrix_to_params(L)[0][0].cpu()), g
            gram, want = res.lattice[g] @ res.lattice[g].T, lats[g] @ lats[g].T
            assert np.abs(gram - want).max() <= 1e-10 * np.abs(want).max(), g
    assert free_rows.any() and not np.array_equal(res.frac_x[free_rows], free_run.frac_x[free_rows])
    # the engine drops the condition for the next call
    assert _crystals(m.sample(None, G, **kw)) == _crystals(free_run)


def _world2(rank):
    from test_gpu_constrained_sampling import _world2 as w
    return w(rank)


@pytest.mark.parametrize("case", ["sites+compositions", "sites+elements", "lattice+compositions"])
def test_keyed_conditioned_crystals_do_not_depend_on_the_batch(device, weights_npz, monkeypatch, case):
    """T = 11, keyed: a conditioned crystal is the same bits in a batch of 300 and in a permuted batch of 17, with the
    CUDA graph on and off, and over two emulated ranks of generate_n_crystals."""
    import arreau_b200.generate as gen
    from arreau_b200.tools.atomic_number_table import ATOMIC_NUMBER
    from test_gpu_constrained_sampling import _systems
    from test_gpu_keyed_sampling import _population
    from test_gpu_wrapper import _model
    m = _model(device, weights_npz, T=11, precision="fp16")
    n = 300
    ids, counts = _population(n, 30)
    rng = np.random.default_rng(31)
    comps = [rng.integers(1, Z, c) for c in counts]
    systems = _systems(n, 32)
    if case == "sites+compositions":
        per = dict(compositions=comps, sites=_sites(counts, rng, comps))
    elif case == "sites+elements":
        per = dict(elements=systems, sites=_sites(counts, rng))
    else:
        per = dict(compositions=comps, lattices=_lattices(n, rng))

    def sample(idx, graph):
        kw = {k: [v[i] for i in idx] for k, v in per.items()}
        if "compositions" not in kw:
            kw["num_atoms"] = torch.as_tensor(counts[idx])
        return m.sample(None, len(idx), crystal_ids=torch.as_tensor(ids[idx]), seed=6, device=device,
                        cuda_graph=graph, **kw)
    sel = np.random.default_rng(33).permutation(n)[:17]
    runs = {}
    for graph in (False, True):
        for name, idx in (("big", np.arange(n)), ("small", sel)):
            res = sample(idx, graph)
            runs[(graph, name)] = _crystals(res)
            if "elements" in per:           # free atoms are in the system; sites keep their own elements
                off = np.concatenate([[0], np.cumsum(res.num_atoms)])
                for j, i in enumerate(idx):
                    k = 0 if per["sites"][i] is None else len(per["sites"][i][0])
                    free_z = set(res.atomic_numbers[off[j] + k:off[j + 1]].tolist())
                    assert free_z <= {ATOMIC_NUMBER[e] for e in systems[i]}, i
    assert runs[(True, "big")] == runs[(False, "big")] and runs[(True, "small")] == runs[(False, "small")]
    for j, g in enumerate(sel):
        assert runs[(False, "small")][j] == runs[(False, "big")][g], g
    # generate_n_crystals: ids are the run's indices, so compare its whole run with two emulated ranks
    gkw = dict(per)
    if "compositions" not in gkw:
        gkw["num_atoms"] = counts
    run = lambda b: gen.generate_n_crystals(m, n, None, device=device, seed=9, keyed_noise=True,  # noqa: E731
                                            num_crystals_per_batch=b, **gkw)
    whole = run(1000)
    shards = []
    for r in range(2):
        monkeypatch.setattr(gen, "dist", _world2(r))
        shards.append(run(64))
    monkeypatch.undo()
    assert _crystals(shards[0]) + _crystals(shards[1]) == _crystals(whole)
    if "compositions" in per:
        assert np.array_equal(whole.atomic_numbers, np.concatenate(comps))
