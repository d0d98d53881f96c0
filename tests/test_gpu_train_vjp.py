"""The hand-written training backward (arreau_ponita_backward, and arreau_ponita_forward_train on the TF32 path) against
the oracle's fp64 vector-Jacobian product (oracle/training.py: ponita_vjp), output by output and block by block.

A gradient reduced to one number per tensor is dominated by the lattice term: a wrong score read-out or a dropped score
contribution to dh would stay far below the tensor's tolerance.  So every check here runs four cotangent sets through
the same forward -- dscore alone, dlogits alone, dlen0 alone (seeded N(0, 1) in fp32, the oracle gets the same values),
and the loss's own output gradients -- and compares the gradient block by block (oracle.training.gradient_blocks: each
read-out row group by the output it produces, x_embedder's scalar and vector columns, every other tensor whole) with
one measure, max|gpu - ref| / max|ref| over the block: 2e-3 on the fp32 path, 0.5 on the TF32 path (GRAD_TOL).  A block whose
reference is identically zero (the read-out rows of an output whose cotangent is zero, the edge chain of a graph
without edges) must be exactly zero.

The engine runs the way TrainEngine.loss_and_grads does (set_batch, noise_batch, predict, compute_loss, backward); the
oracle gets the noised state and the per-atom timesteps the GPU produced, and the GPU's edge list must equal the
oracle graph's first, so that a graph difference is reported as one.  Topologies: the C5 training batch (270 crystals,
~2 500 atoms), a ragged batch (a 236-atom crystal, 1-atom crystals, atoms without any neighbour), receiver rows longer
than 8 (cap 12), an uncapped graph whose edge buffers grow, r = 7, and a batch without a single edge."""
import numpy as np
import pytest
import torch

from conftest import TOL_FP32, f64_default

pytestmark = pytest.mark.gpu
T, Z, F, V = 1000, 90, 164, 4
# DESIGN.md section 6: a block whose exact value is a sum over the orientation grid of terms that nearly cancel (the
# score row, x_embedder's vector columns, and under the score's cotangent most of the network) keeps TF32's operand
# rounding of 2^-11 times the un-cancelled magnitude
GRAD_TOL = {"fp32": 2e-3, "tf32": 0.5}
TOL_TF32_FORWARD = 5e-3        # DESIGN.md section 6: score, logits, len0 of arreau_ponita_forward_train, of max|ref|
COTANGENTS = ("dscore", "dlogits", "dlen0", "loss")
SLICE_CRYSTALS = 45


# --------------------------------------------------------------------------------------------- topologies
def _concat(parts):
    from arreau_b200.synthetic import Crystals
    return Crystals(*(np.concatenate([getattr(c, k) for c in parts]) for k in ("frac", "types", "lengths", "angles",
                                                                                  "num_atoms")))


def _sparse(num, lo, hi, seed, volume_per_atom):
    """make_crystals geometry scaled to `volume_per_atom` A^3 per atom (the data set's density is ~18 A^3)."""
    from arreau_b200.synthetic import VOLUME_PER_ATOM, make_crystals
    cr = make_crystals(num, lo, hi, seed=seed)
    cr.lengths = cr.lengths * np.cbrt(volume_per_atom / VOLUME_PER_ATOM)
    return cr


def _t(rng, n, hi=T):
    return rng.integers(1, hi + 1, size=n)


def _batch_c5(rng):
    from arreau_b200.synthetic import make_training_batch
    cr = make_training_batch(270, seed=0)
    return cr, _t(rng, cr.num_crystals)


def _take(cr, first, stop):
    """Crystals first..stop-1 of `cr`."""
    a0, a1 = int(cr.num_atoms[:first].sum()), int(cr.num_atoms[:stop].sum())
    return type(cr)(cr.frac[a0:a1], cr.types[a0:a1], cr.lengths[first:stop], cr.angles[first:stop], cr.num_atoms[first:stop])


def _batch_ragged(rng):
    """Crystals that keep their geometry (isolated atoms, 1-atom cells) are noised at t <= 50, where the lattice moves
    by < 8 % of eps; the others at any t."""
    from arreau_b200.synthetic import make_crystals
    ordinary, big, single = make_crystals(16, 2, 40, seed=21), make_crystals(1, 236, seed=22), make_crystals(6, 1, seed=23)
    lonely = _sparse(6, 1, 3, seed=24, volume_per_atom=1000.0)
    parts = [(_take(ordinary, 0, 8), T), (_take(single, 0, 3), 50), (big, T), (lonely, 50),
             (_take(single, 3, 6), 50), (_take(ordinary, 8, 16), T)]
    return _concat([c for c, _ in parts]), np.concatenate([_t(rng, c.num_crystals, hi) for c, hi in parts])


def _batch_no_edges(rng):
    """1-atom cells of ~2000 A^3 and 2-atom body-centred cells of ~4000 A^3: the nearest image or partner is > 9 A
    away; t <= 50 keeps the lattices."""
    one = _sparse(12, 1, None, seed=31, volume_per_atom=2000.0)
    two = _sparse(4, 2, None, seed=32, volume_per_atom=2000.0)
    two.frac = np.tile(np.array([[0.1, 0.2, 0.3], [0.6, 0.7, 0.8]]), (4, 1))
    cr = _concat([one, two])
    return cr, _t(rng, cr.num_crystals, 50)


def _batch_mixed(num, hi, seed, t_hi=T):
    def build(rng):
        from arreau_b200.synthetic import make_crystals
        cr = make_crystals(num, 1, hi, seed=seed)
        return cr, _t(rng, cr.num_crystals, t_hi)
    return build


# name -> (batch builder, radius, cap, what the graph must show)
TOPOLOGIES = {
    "c5": (_batch_c5, 5.0, 8, lambda g: g["N"] > 2000 and g["G"] == 270),
    "ragged": (_batch_ragged, 5.0, 8, lambda g: g["max_atoms"] == 236 and g["isolated"] > 0 and g["min_atoms"] == 1),
    "cap12": (_batch_mixed(24, 40, 41), 5.0, 12, lambda g: g["max_deg"] > 8),
    "uncapped": (_batch_mixed(12, 30, 42, t_hi=600), 5.0, 0, lambda g: g["E"] > 32 * g["N"]),
    "r7": (_batch_mixed(24, 40, 43), 7.0, 8, lambda g: g["E"] > 0),
    "no_edges": (_batch_no_edges, 5.0, 8, lambda g: g["E"] == 0),
}


def _make_batch(name):
    from oracle import restatement as R
    build, radius, cap, _ = TOPOLOGIES[name]
    rng = np.random.default_rng(sorted(TOPOLOGIES).index(name) + 100)
    cr, timestep = build(rng)
    G, N = cr.num_crystals, cr.total_atoms
    with f64_default():
        lattice0 = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
    return dict(cr=cr, radius=radius, cap=cap,
                args=(cr.frac, cr.types, lattice0, timestep, rng.standard_normal((N, 3)), rng.random((N, Z)),
                      rng.standard_normal((G, 3))),
                cot=dict(dscore=rng.standard_normal((N, 3)).astype(np.float32),
                         dlogits=rng.standard_normal((N, Z)).astype(np.float32),
                         dlen0=rng.standard_normal((G, 3)).astype(np.float32)))


# --------------------------------------------------------------------------------------------- engine
def _engine(device, weights_npz, num_atoms, radius, cap, precision, node_capacity=None, crystal_capacity=None):
    from arreau_b200.tables import build_tables
    from arreau_b200.training import FlatParams, TrainEngine
    p = FlatParams(F, V, Z, device)
    p.load_state_dict({k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")})
    return TrainEngine(p, build_tables(T, Z), weights_npz["fourier_w"], weights_npz["ori_grid"], num_atoms, radius, cap,
                       device=device, backward_precision=precision, node_capacity=node_capacity,
                       crystal_capacity=crystal_capacity)


def _forward(te, b):
    """loss_and_grads up to the backward."""
    te.repack()
    te.set_batch(*b["args"])
    te.noise_batch()
    te.predict()
    te.compute_loss()


def _backward(te, b, cot):
    """The parameter gradients (a copy) for one cotangent set: the loss's own, or one output's seeded cotangent alone."""
    if cot == "loss":
        return te.backward().clone()
    out = {k: torch.zeros_like(getattr(te, k)) for k in ("dscore", "dlogits", "dlen0")}
    out[cot] = torch.as_tensor(b["cot"][cot]).to(te.device)
    return te.backward(**out).clone()


# --------------------------------------------------------------------------------------------- the oracle, once per topology
@pytest.fixture(scope="module")
def case(device, weights_npz):
    """name -> the batch, what both precision engines computed from it, and the oracle's fp64 outputs and gradients
    for every cotangent set (the loss's own cotangents are each precision's own).  Cached for the module."""
    from oracle import restatement as R, training as TR
    cache = {}

    def get(name):
        if name in cache:
            return cache[name]
        b = _make_batch(name)
        cr = b["cr"]
        gpu = {}
        for prec in ("fp32", "tf32"):
            te = _engine(device, weights_npz, cr.num_atoms, b["radius"], b["cap"], prec)
            _forward(te, b)
            e = te.eng
            torch.cuda.synchronize()
            assert int(e.overflow_flag.item()) == 0
            E = e.num_edges()
            gpu[prec] = dict(
                state=[x.cpu().numpy() for x in (e.frac, e.types, te.t_atom, e.lengths, e.angles, e.lattice)],
                edges=np.stack([e.src[:E].cpu().numpy(), e.dst[:E].cpu().numpy()]).astype(np.int64),
                cell=e.cell[:E].cpu().numpy().astype(np.int64),
                out=dict(score=e.score.cpu().numpy(), logits=e.logits.cpu().numpy(), len0=e.len0.cpu().numpy()),
                loss=te.loss.cpu().numpy(), loss_cot=[x.cpu().numpy().copy() for x in (te.dscore, te.dlogits, te.dlen0)])
        for a, c in zip(gpu["fp32"]["state"], gpu["tf32"]["state"]):
            assert np.array_equal(a, c)            # noising is fp64 and does not depend on the network's precision
        frac, types, t_atom, lengths, angles, lattice = gpu["fp32"]["state"]
        deg = np.bincount(gpu["fp32"]["edges"][1], minlength=cr.total_atoms)
        stats = dict(N=cr.total_atoms, G=cr.num_crystals, E=int(deg.sum()), max_deg=int(deg.max(initial=0)),
                     isolated=int((deg == 0).sum()), max_atoms=int(cr.num_atoms.max()), min_atoms=int(cr.num_atoms.min()))
        assert TOPOLOGIES[name][3](stats), (name, stats)
        c = b["cot"]
        cots = {"dscore": (c["dscore"], None, None), "dlogits": (None, c["dlogits"], None),
                "dlen0": (None, None, c["dlen0"]), "loss/fp32": gpu["fp32"]["loss_cot"], "loss/tf32": gpu["tf32"]["loss_cot"]}
        T64 = lambda a: None if a is None else torch.as_tensor(np.asarray(a), dtype=torch.float64)  # noqa: E731
        with f64_default():
            sd = {k: T64(weights_npz[k]) for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
            W = R.PonitaWeights(sd, T64(weights_npz["ori_grid"]), b["radius"])
            # the GPU's lattice: mirror images tie exactly, the cap's choice between them rests on its last bit
            outs, grads, (ei, cell_off) = TR.ponita_vjp(
                W, R.DiffusionTables.build(T, Z), T64(weights_npz["fourier_w"]), T64(frac), torch.as_tensor(types),
                torch.as_tensor(t_atom), torch.as_tensor(cr.num_atoms), T64(lengths), T64(angles), b["radius"], b["cap"],
                [tuple(T64(x) for x in v) for v in cots.values()], slice_crystals=SLICE_CRYSTALS, lattice=T64(lattice))
        assert ei.shape[1] == stats["E"], f"{name}: GPU graph has {stats['E']} edges, the oracle's {ei.shape[1]}"
        assert np.array_equal(gpu["fp32"]["edges"], ei.numpy()), f"{name}: GPU edge list differs from the oracle graph"
        img = gpu["fp32"]["cell"]    # index into itertools.product((-1, 0, 1), repeat=3); the oracle gives -cell
        cells = np.stack([img // 9 - 1, img // 3 % 3 - 1, img % 3 - 1], 1)
        assert np.array_equal(cells, -cell_off.numpy().astype(np.int64)), \
            f"{name}: GPU edge images differ from the oracle graph's"
        print(f"\n{name}: N={stats['N']} G={stats['G']} E={stats['E']} E/N={stats['E'] / stats['N']:.1f} "
              f"max receiver row {stats['max_deg']}, {stats['isolated']} atoms without a neighbour")
        cache[name] = dict(b=b, gpu=gpu, outs={k: v.numpy() for k, v in outs.items()},
                           grads={k: {p: g.numpy() for p, g in gr.items()} for k, gr in zip(cots, grads)})
        return cache[name]
    return get


def block_errors(got: dict, ref: dict) -> dict:
    """block name -> max|got - ref| / max|ref| over the block; a block whose reference is identically zero gives 0 when
    the GPU's is exactly zero too and inf otherwise."""
    from oracle import training as TR
    out = {}
    for block, parts in TR.gradient_blocks({k: v.shape for k, v in ref.items()}, Z, F):
        g = np.concatenate([np.asarray(got[k], dtype=np.float64)[idx].ravel() for k, idx in parts])
        r = np.concatenate([ref[k][idx].ravel() for k, idx in parts])
        m = np.abs(r).max()
        out[block] = float(np.abs(g - r).max() / m) if m > 0 else (0.0 if not np.any(g) else float("inf"))
    return out


# --------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("cot", COTANGENTS)
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("topology", list(TOPOLOGIES))
def test_backward_blocks_against_oracle(device, weights_npz, case, topology, precision, cot):
    c = case(topology)
    b = c["b"]
    te = _engine(device, weights_npz, b["cr"].num_atoms, b["radius"], b["cap"], precision)
    _forward(te, b)
    if cot == "loss":       # the same forward as the fixture's: the same output gradients
        for got, ref in zip((te.dscore, te.dlogits, te.dlen0), c["gpu"][precision]["loss_cot"]):
            assert np.array_equal(got.cpu().numpy(), ref)
    grad = _backward(te, b, cot)
    got = {k: v.cpu().numpy() for k, v in te.p._views(grad).items()}
    errs = block_errors(got, c["grads"][f"loss/{precision}" if cot == "loss" else cot])
    worst = max(errs, key=errs.get)
    print(f"{topology} {precision} {cot}: worst block {worst} {errs[worst]:.2e}")
    bad = {k: v for k, v in errs.items() if not v < GRAD_TOL[precision]}
    assert not bad, bad


@pytest.mark.parametrize("topology", list(TOPOLOGIES))
def test_forward_outputs_against_oracle(device, case, topology):
    """score, logits and len0 of both training forwards (the plain fp32 forward: 1e-4; arreau_ponita_forward_train on
    the TF32 path: its stated bound) against the oracle's, output by output."""
    c = case(topology)
    errs = {}
    for prec, tol in (("fp32", TOL_FP32), ("tf32", TOL_TF32_FORWARD)):
        for k in ("score", "logits", "len0"):
            ref, got = c["outs"][k], c["gpu"][prec]["out"][k]
            errs[prec, k] = float(np.abs(got - ref).max() / np.abs(ref).max())
            assert errs[prec, k] < tol, (prec, k, errs[prec, k])
    print(f"{topology} forward: " + ", ".join(f"{p} {k} {v:.2e}" for (p, k), v in errs.items()))


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_capacity_engine_rebound_from_a_denser_batch(device, weights_npz, case, precision):
    """A capacity engine that has just run the C5 batch, re-bound to the ragged batch and to the batch without edges:
    its edge slab rows between E and the capacity still hold the C5 batch's data.  Every gradient must be bit-identical
    to a fresh engine's."""
    c5 = case("c5")["b"]
    shared = _engine(device, weights_npz, c5["cr"].num_atoms, 5.0, 8, precision,
                     node_capacity=c5["cr"].total_atoms, crystal_capacity=c5["cr"].num_crystals)
    _forward(shared, c5)
    assert float(_backward(shared, c5, "loss").abs().max()) > 0
    for name in ("ragged", "no_edges"):
        b = case(name)["b"]
        assert (b["radius"], b["cap"]) == (5.0, 8)
        fresh = _engine(device, weights_npz, b["cr"].num_atoms, 5.0, 8, precision)
        shared.set_topology(b["cr"].num_atoms)
        for cot in COTANGENTS:
            _forward(shared, b)
            _forward(fresh, b)
            assert torch.equal(shared.loss, fresh.loss), (name, cot)
            assert torch.equal(_backward(shared, b, cot), _backward(fresh, b, cot)), (name, cot)
