"""Uniqueness and novelty on the host: a numpy fit oracle of arreau_structure_fit_pairs, a literal restatement of
pymatgen's group_structures checked against the greedy resolution of inference/structure_match.py, key grouping and
pair lists, the summary, the C ABI argument checks and the refusal of crystal_metrics --unique_novel.

The oracle is match_pair of test_structure_match_host.py with pymatgen's fit objective (StructureMatcher._match with
use_rms=False, break_on_match=True): a candidate's value is its largest normalised distance, the pair is matched at
the first candidate below stol, in the kernel's enumeration order (mappings by band index, then translations)."""
import ctypes as C
import itertools
import json

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from test_structure_match_host import (BAND_CAP, COMPOSITION, DEGENERATE, MATCHED, MAX_ATOMS, MAX_STEPS,
                                       SEARCH_LIMIT, TOO_LARGE, _IMAGES, _recip, from_params, int_inv, lll_reduce,
                                       match_pair, niggli_reduce, params, random_cell, transformed_copy, wrap)


def _fit_result(flags, max_dist=np.nan, num_mappings=0):
    return dict(max_dist=max_dist, num_mappings=num_mappings, flags=flags)


def fit_pair(f1, L1, z1, f2, L2, z2, stol=0.3, ltol=0.2, angle_tol=5.0):
    """max_dist, num_mappings and flags of fit(crystal 1, crystal 2); crystal 1's lattice is the one mapped."""
    f1, f2 = np.asarray(f1, np.float64).reshape(-1, 3), np.asarray(f2, np.float64).reshape(-1, 3)
    z1, z2 = np.asarray(z1, np.int64).reshape(-1), np.asarray(z2, np.int64).reshape(-1)
    o1, o2 = np.argsort(z1, kind="stable"), np.argsort(z2, kind="stable")
    f1, z1, f2, z2 = f1[o1], z1[o1], f2[o2], z2[o2]
    n = len(z1)
    if len(z2) != n or np.any(z1 != z2):
        return _fit_result(COMPOSITION)
    if n > MAX_ATOMS:
        return _fit_result(TOO_LARGE)
    L1, L2 = np.asarray(L1, np.float64), np.asarray(L2, np.float64)
    if n == 0 or not (np.isfinite(L1).all() and np.isfinite(L2).all() and np.isfinite(f1).all()
                      and np.isfinite(f2).all()):
        return _fit_result(DEGENERATE)
    if not (abs(np.linalg.det(L1)) >= 0.1 and abs(np.linalg.det(L2)) >= 0.1):
        return _fit_result(DEGENERATE)
    N1, C1, ok1 = niggli_reduce(L1)
    N2, C2, ok2 = niggli_reduce(L2)
    if not (ok1 and ok2):
        return _fit_result(DEGENERATE)
    f1n, f2n = wrap(f1 @ int_inv(C1)), wrap(f2 @ int_inv(C2))
    ratio = (abs(np.linalg.det(N2)) / abs(np.linalg.det(N1))) ** (1.0 / 6.0)
    L1s, L2s = N1 * ratio, N2 / ratio
    p2 = params(L2s)
    K = np.floor(p2[:3].max() * (1 + ltol) * _recip(L1s))
    if not np.all(K <= MAX_STEPS):
        return _fit_result(SEARCH_LIMIT)
    grid = np.array(list(itertools.product(*[np.arange(-k, k + 1) for k in K])), dtype=np.float64)
    v = grid @ L1s
    d = np.sqrt((v * v).sum(1))
    bands = []
    for length in p2[:3]:
        q = d / length
        sel = np.nonzero((q < 1 + ltol) & (q > 1 / (1 + ltol)))[0]
        if len(sel) > BAND_CAP:
            return _fit_result(SEARCH_LIMIT)
        bands.append(sel)

    def within(i, j, target):
        x = np.clip((v[i] @ v[j].T) / d[i][:, None] / d[j][None, :], -1, 1)
        return np.abs(np.arccos(x) * 180.0 / np.pi - target) < angle_tol

    A, B, Cb = bands
    alpha, beta, gamma = within(B, Cb, p2[3]), within(A, Cb, p2[4]), within(A, B, p2[5])
    blocks = np.concatenate([[0], np.nonzero(np.diff(z2))[0] + 1, [n]])
    rare = int(np.argmin(np.diff(blocks)))
    anchor, t_sites = blocks[rare], np.arange(blocks[rare], blocks[rare + 1])
    same = z1[None, :] == z2[:, None]
    best, num_mappings = np.inf, 0
    for i in range(len(A)):
        for j in range(len(B)):
            if not gamma[i, j]:
                continue
            for k in range(len(Cb)):
                if not (alpha[j, k] and beta[i, k]):
                    continue
                S = grid[[A[i], B[j], Cb[k]]]
                if abs(round(np.linalg.det(S))) != 1:
                    continue
                num_mappings += 1
                for val in _candidates(S, v[[A[i], B[j], Cb[k]]], f1n, f2n, p2, n, stol, blocks, anchor, t_sites,
                                       same):
                    best = min(best, val)
                    if val < stol:
                        return _fit_result(MATCHED, val, num_mappings)
    return _fit_result(0, best if np.isfinite(best) else np.nan, num_mappings)


def _candidates(S, M, f1n, f2n, p2, n, stol, blocks, anchor, t_sites, same):
    """max(dist) of every translation of one lattice mapping that passes the prefilter and has a complete matching,
    in translation order."""
    fc1 = wrap(f1n @ int_inv(S))
    avg = from_params((params(M) + p2) / 2)
    norm = (n / abs(np.linalg.det(avg))) ** (1.0 / 3.0)
    frac_tol = 2 * stol * _recip(avg) / norm
    Bl, Mp, _ = lll_reduce(avg)
    lll_tol = 2 * stol * _recip(Bl) / norm
    Mpinv = int_inv(Mp)
    lf1 = wrap(fc1 @ Mpinv)
    im = _IMAGES @ Bl
    for t in fc1[t_sites] - f2n[anchor]:
        dd = (f2n + t)[:, None, :] - fc1[None, :, :]
        if not np.all(np.any(np.all(np.abs(dd - np.round(dd)) <= frac_tol, axis=-1) & same, axis=1)):
            continue
        lf2 = wrap((f2n + t) @ Mpinv)
        vecs = np.empty((n, 3))
        feasible = True
        for b0, b1 in zip(blocks[:-1], blocks[1:]):
            D = lf1[None, b0:b1] - lf2[b0:b1, None]
            adm = np.all(np.abs(D - np.round(D)) <= lll_tol, axis=-1)
            cart = (D @ Bl)[:, :, None, :] + im[None, None]
            d2 = (cart * cart).sum(-1)
            kbest = np.argmin(d2, axis=-1)
            cost = np.where(adm, np.take_along_axis(d2, kbest[..., None], -1)[..., 0], np.inf)
            try:
                rows, cols = linear_sum_assignment(cost)
            except ValueError:
                feasible = False
                break
            vecs[b0 + rows] = cart[rows, cols, kbest[rows, cols]]
        if feasible:
            yield (np.sqrt(((vecs - vecs.mean(0)) ** 2).sum(1)) * norm).max()


def _crystal(inputs, g):
    off = np.concatenate([[0], np.cumsum(inputs[3])])
    return inputs[0][off[g]:off[g + 1]], inputs[1][g], inputs[2][off[g]:off[g + 1]]


def fit_pairs(set1, set2, index1, index2, **kw):
    """fit_pair over the pairs (index1[p], index2[p]) of two (frac, lattice, z, num_atoms) tuples; an index outside
    its set is DEGENERATE.  Arrays max_dist, num_mappings, flags."""
    out = []
    for a, b in zip(np.asarray(index1).reshape(-1), np.asarray(index2).reshape(-1)):
        if not (0 <= a < len(set1[3]) and 0 <= b < len(set2[3])):
            out.append(_fit_result(DEGENERATE))
        else:
            out.append(fit_pair(*_crystal(set1, a), *_crystal(set2, b), **kw))
    return {k: np.array([o[k] for o in out], dtype=np.float64 if k == "max_dist" else np.int64)
            for k in ("max_dist", "num_mappings", "flags")}


def group_structures(considered, keys, fit):
    """pymatgen's StructureMatcher.group_structures, literally: the considered crystals stably sorted by key, and
    within each key the first unmatched crystal takes every unmatched crystal u with fit(it, u).  Lists of indices."""
    s_list = [i for i in range(len(considered)) if considered[i]]
    groups = []
    for _, g in itertools.groupby(sorted(s_list, key=lambda i: keys[i]), key=lambda i: keys[i]):
        unmatched = list(g)
        while unmatched:
            ref = unmatched.pop(0)
            inds = [k for k in range(len(unmatched)) if fit(ref, unmatched[k])]
            groups.append([ref] + [unmatched[k] for k in inds])
            unmatched = [unmatched[k] for k in range(len(unmatched)) if k not in inds]
    return groups


def groups_of(group):
    """The partition a group array describes, as group_structures lists it (sorted for comparison)."""
    out = {}
    for i, r in enumerate(group):
        if r >= 0:
            out.setdefault(int(r), []).append(i)
    return sorted(out.values())


def _pack(crystals):
    return (np.concatenate([np.asarray(c[0], np.float64).reshape(-1, 3) for c in crystals]),
            np.stack([np.asarray(c[1], np.float64) for c in crystals]),
            np.concatenate([np.asarray(c[2], np.int64).reshape(-1) for c in crystals]),
            np.array([len(c[2]) for c in crystals], np.int64))


def _metrics(flags):
    from arreau_b200.inference.crystal_metrics import CrystalMetrics
    G = len(flags)
    return CrystalMetrics(num_atoms=np.ones(G, np.int64), volume=np.ones(G), min_dist=np.ones(G),
                          density=np.ones(G), num_elements=np.ones(G, np.int32), flags=np.asarray(flags, np.int32))


# ---- the oracle ------------------------------------------------------------------------------------------------------
def test_fit_oracle_on_copies_and_against_the_rms_oracle():
    rng = np.random.default_rng(0)
    for k in range(24):
        n = int(rng.integers(2, 10))
        f, L, z = rng.random((n, 3)), random_cell(rng, n), rng.integers(1, 4, n)
        if k % 3 == 2:                                       # same composition, random positions
            g = (rng.random((n, 3)), L @ np.diag(1 + 0.05 * rng.standard_normal(3)), z[rng.permutation(n)])
        else:
            g = transformed_copy(f, L, z, rng, sigma=(0.0, 0.02)[k % 3])
        r = fit_pair(*g, f, L, z)
        m = match_pair(*g, f, L, z, stol=0.3, ltol=0.2, angle_tol=5.0)
        if k % 3 != 2:
            assert r["flags"] == MATCHED and r["max_dist"] < 0.3
        if k % 3 == 0:
            assert r["max_dist"] <= 1e-10
        if r["flags"] == MATCHED:                            # rms <= max: fit implies an rms match
            assert m["flags"] == MATCHED and m["rms"] <= r["max_dist"] + 1e-12
            assert r["num_mappings"] <= m["num_mappings"]
        else:                                                # the whole search ran
            assert r["num_mappings"] == m["num_mappings"]
            assert not np.isfinite(r["max_dist"]) or r["max_dist"] >= m["max_dist"] - 1e-12


def test_fit_oracle_flags():
    L = np.array([[3.0, 0, 0], [0.2, 3.1, 0], [0.3, -0.2, 12.0]])
    f = np.array([[0.0, 0.0, 0.0], [0.5, 0.5, 0.02], [0.0, 0.5, 0.5], [0.5, 0.0, 0.53]])
    z = np.array([8, 8, 26, 26])
    assert fit_pair(f, L, z, f, L, z)["flags"] == MATCHED
    assert fit_pair(f, L, [8, 8, 26, 27], f, L, z)["flags"] == COMPOSITION
    assert fit_pair(f, np.full((3, 3), np.nan), z, f, L, z)["flags"] == DEGENERATE
    r = fit_pairs(_pack([(f, L, z)]), _pack([(f, L, z)]), [0, 1, -1], [0, 0, 0])
    assert r["flags"].tolist() == [MATCHED, DEGENERATE, DEGENERATE]


# ---- group_structures and the greedy resolution ----------------------------------------------------------------------
def test_greedy_resolution_is_group_structures():
    from arreau_b200.inference.structure_match import composition_keys, resolve_groups, uniqueness_pairs
    rng = np.random.default_rng(1)
    for trial in range(200):
        G = int(rng.integers(0, 40))
        na = rng.integers(1, 4, G)
        z = rng.integers(1, 3, int(na.sum()))
        considered = rng.random(G) < 0.85
        keys = composition_keys(z, na)
        rel = rng.random((G, G)) < (0.1, 0.4, 0.9)[trial % 3]            # any relation: not symmetric or transitive
        i1, i2 = uniqueness_pairs(keys, considered)
        group = resolve_groups(considered, i1, i2, rel[i1, i2])
        expect = group_structures(considered, keys, lambda a, b: rel[a, b])
        assert groups_of(group) == sorted(expect)
        for g in expect:                                                  # the representative is the first member
            assert all(group[i] == g[0] for i in g)
        assert np.all(group[~considered] == -1)


def test_keys_and_pair_lists():
    from arreau_b200.inference.structure_match import (composition_keys, novelty_pairs, reduced_formula,
                                                       resolve_groups, uniqueness_pairs)
    assert composition_keys(np.zeros(0), np.zeros(0)) == []
    e = uniqueness_pairs([], np.zeros(0, np.bool_))
    assert e[0].shape == (0,) and e[1].shape == (0,)
    assert resolve_groups(np.zeros(0, np.bool_), *e, np.zeros(0, np.bool_)).shape == (0,)
    one = composition_keys([8, 26], [2])
    assert len(uniqueness_pairs(one, [True])[0]) == 0
    assert resolve_groups(np.array([True]), *uniqueness_pairs(one, [True]), np.zeros(0, np.bool_)).tolist() == [0]
    # crystals: Fe O | O Fe | Fe O O | O Fe (atom count 2) | Fe O with an unknown atom | O Fe
    z = [26, 8, 8, 26, 26, 8, 8, 8, 26, 26, 8, 2001, 8, 26]
    na = [2, 2, 3, 2, 3, 2]
    keys = composition_keys(z, na)
    assert keys[0] == keys[1] == keys[3] == keys[5] and keys[2] != keys[0] and keys[4] != keys[0]
    considered = np.array([True, True, True, False, False, True])        # 3 not valid, 4 has an unknown element
    i1, i2 = uniqueness_pairs(keys, considered)
    assert sorted(zip(i1.tolist(), i2.tolist())) == [(0, 1), (0, 5), (1, 5)]
    ref_keys = composition_keys([8, 26, 26, 8, 8, 26, 8, 8, 26, 26, 8, 8], [2, 3, 3, 4])
    n1, n2 = novelty_pairs(keys, considered, ref_keys)
    assert sorted(zip(n1.tolist(), n2.tolist())) == [(0, 0), (1, 0), (2, 1), (2, 2), (5, 0)]
    assert reduced_formula(ref_keys[3]) == reduced_formula(keys[0]) == ((8, 1), (26, 1))
    assert reduced_formula(ref_keys[1]) == ((8, 2), (26, 1))
    assert len(novelty_pairs(keys, considered, [])[0]) == 0
    fit = {(0, 1): False, (0, 5): True, (1, 5): True}
    group = resolve_groups(considered, i1, i2, np.array([fit[p] for p in zip(i1.tolist(), i2.tolist())]))
    assert group.tolist() == [0, 1, 2, -1, -1, 0]
    with pytest.raises(ValueError, match="index1 < index2"):
        resolve_groups(considered, [1], [0], [True])


def _fake_fit(monkeypatch):
    """structure_fit_pairs replaced by the numpy oracle, so unique_novel runs on the host."""
    from arreau_b200.inference import structure_match as sm

    def fake(set1, set2, index1, index2, stol=0.3, ltol=0.2, angle_tol=5.0, device="cuda", max_chunk_pairs=0):
        r = fit_pairs(set1, set2, index1, index2, stol=stol, ltol=ltol, angle_tol=angle_tol)
        return sm.FitPairs(matched=(r["flags"] & MATCHED) != 0, max_dist=r["max_dist"],
                           num_mappings=r["num_mappings"].astype(np.int32), flags=r["flags"].astype(np.int32))
    monkeypatch.setattr(sm, "structure_fit_pairs", fake)
    return sm


def test_unique_novel_with_the_oracle(monkeypatch):
    sm = _fake_fit(monkeypatch)
    rng = np.random.default_rng(2)
    bases = []
    for k in range(6):                      # three compositions, two structures each
        n = 5 + k // 2
        z = np.array([8] * (n - 2) + [26, 12])
        bases.append((rng.random((n, 3)), random_cell(rng, n), z))
    order = [0, 1, 2, 0, 3, 4, 5, 1, 3, 0, 5]
    gen = [transformed_copy(*bases[b], rng, sigma=(0.0, 0.02)[k % 2]) for k, b in enumerate(order)]
    gen.append((bases[0][0], bases[0][1], np.where(np.arange(5) == 0, 2001, bases[0][2])))   # unknown element
    g = _pack(gen)
    # the reference: bases 0 and 2 transformed again, and an O2 Fe crystal; bases 4 and 5 (O5 Fe Mg) have no formula
    # in it
    ref = _pack([transformed_copy(*bases[b], rng, sigma=0.02) for b in (0, 2)]
                + [(rng.random((3, 3)), random_cell(rng, 3), [8, 8, 26])])
    flags = np.ones(len(gen), np.int32)
    flags[-1] = 2                                                        # UNKNOWN_ELEMENT
    un = sm.unique_novel(g, _metrics(flags), ref)
    expect = {}
    for i, b in enumerate(order):
        expect.setdefault(b, []).append(i)
    assert groups_of(un.group) == sorted(expect.values())
    assert un.group[-1] == -1 and not un.unique[-1] and not un.novel[-1]
    assert un.novel[:-1].tolist() == [b not in (0, 2) for b in order]
    assert un.new_formula[:-1].tolist() == [b in (4, 5) for b in order]
    keys = sm.composition_keys(g[2], g[3])
    fit = lambda a, b: fit_pair(*_crystal(g, a), *_crystal(g, b))["flags"] == MATCHED  # noqa: E731
    assert groups_of(un.group) == sorted(group_structures(un.considered, keys, fit))
    s = sm.unique_novel_summary(un)
    G = len(gen)
    assert (s["num_considered"], s["num_unique"], s["num_novel"], s["num_unique_novel"]) == (G - 1, 6, 7, 4)
    assert s["frac_unique"] == 6 / G and s["frac_novel"] == 7 / G and s["frac_unique_novel"] == 4 / G
    assert s["num_new_formula"] == 3
    assert s["num_fit_pairs"] == len(un.uniqueness_fit.flags) + len(un.novelty_fit.flags)
    json.dumps(s)


def test_summary_counts():
    from arreau_b200.inference.structure_match import FitPairs, UniqueNovel, unique_novel_summary
    fl = lambda f: FitPairs(matched=(np.asarray(f, np.int32) & 1) != 0, max_dist=np.zeros(len(f)),  # noqa: E731
                            num_mappings=np.zeros(len(f), np.int32), flags=np.asarray(f, np.int32))
    considered = np.array([True, True, True, True, False, True])
    un = UniqueNovel(considered=considered, group=np.array([0, 0, 2, 3, -1, 2]),
                     unique=np.array([True, False, True, True, False, False]),
                     novel=np.array([True, True, False, True, False, False]),
                     new_formula=np.array([False, False, False, True, False, False]),
                     uniqueness_pairs=(np.array([0, 2]), np.array([1, 5])), uniqueness_fit=fl([1, 1]),
                     novelty_pairs=(np.arange(5), np.zeros(5, np.int64)), novelty_fit=fl([8, 4, 1, 16, 0]))
    s = unique_novel_summary(un)
    assert s == dict(num_considered=5, num_unique=3, frac_unique=0.5, num_novel=3, frac_novel=0.5,
                     num_unique_novel=2, frac_unique_novel=2 / 6, num_new_formula=1, num_fit_pairs=7,
                     num_fit_search_limit=1, num_fit_degenerate=1, num_fit_too_large=1)
    un.novel = un.new_formula = un.novelty_fit = None
    s = unique_novel_summary(un)
    assert "num_novel" not in s and s["num_fit_pairs"] == 2
    empty = UniqueNovel(considered=np.zeros(0, np.bool_), group=np.zeros(0, np.int64), unique=np.zeros(0, np.bool_),
                        novel=np.zeros(0, np.bool_), new_formula=np.zeros(0, np.bool_),
                        uniqueness_pairs=(np.zeros(0), np.zeros(0)), uniqueness_fit=fl([]),
                        novelty_pairs=(np.zeros(0), np.zeros(0)), novelty_fit=fl([]))
    s = unique_novel_summary(empty)
    assert s["frac_unique"] is None and s["frac_novel"] is None and s["num_fit_pairs"] == 0


# ---- C ABI and CLI ---------------------------------------------------------------------------------------------------
def test_fit_entry_point_argument_validation():
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p)
    args = lambda **kw: [kw.get(k, v) for k, v in (  # noqa: E731
        ("f1", p), ("l1", p), ("z1", p), ("o1", p), ("n1", 4), ("c1", 1), ("f2", p), ("l2", p), ("z2", p), ("o2", p),
        ("n2", 4), ("c2", 1), ("i1", p), ("i2", p), ("g", 1), ("stol", 0.3), ("ltol", 0.2), ("atol", 5.0),
        ("md", p), ("nm", p), ("fl", p), ("stream", None))]
    assert lib.arreau_structure_fit_pairs(*args(g=0, f1=None, l1=None, i1=None, md=None)) == 0
    for k in ("l1", "o1", "l2", "o2", "i1", "i2", "md", "nm", "fl", "f1", "z1", "f2", "z2"):
        assert lib.arreau_structure_fit_pairs(*args(**{k: None})) == -4, k
    assert lib.arreau_structure_fit_pairs(*args(n1=0, f1=None, z1=None, g=-1)) == -1
    for kw in (dict(g=-1), dict(n1=-4), dict(n2=-4), dict(c1=-1), dict(c2=-1), dict(stol=0.0), dict(ltol=-0.2),
               dict(atol=float("nan")), dict(stol=float("inf"))):
        assert lib.arreau_structure_fit_pairs(*args(**kw)) == -1, kw


def test_structure_fit_pairs_host_checks():
    from arreau_b200.inference.structure_match import structure_fit_pairs
    s = _pack([(np.zeros((1, 3)), np.eye(3) * 3, [8])])
    with pytest.raises(ValueError, match="CUDA"):
        structure_fit_pairs(s, s, [0], [0], device="cpu")


def test_unique_novel_cli_refusal(tmp_path, capsys):
    from arreau_b200.inference import crystal_metrics
    with pytest.raises(SystemExit):
        crystal_metrics.main([str(tmp_path / "missing.npz"), "--unique_novel"])
    assert "--unique_novel needs --reference" in capsys.readouterr().err
