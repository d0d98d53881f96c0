"""Structure matcher on the host: a numpy / scipy oracle of arreau_structure_match (inference/structure_match.py), its
analytic checks, the Niggli reduction, the C ABI argument checks and the refusals of crystal_metrics --match.

It restates pymatgen's StructureMatcher.get_rms_dist(generated, source) with scale=True, attempt_supercell=False and
primitive_cell=False, step by step and in plain numpy, independently of the kernel's method: the assignment is
scipy.optimize.linear_sum_assignment on the full cost matrix, the prefilter and the costs are vectorised over all pairs.
The integer steps (LLL, Niggli, the band enumeration order, the mapping order) are the kernel's, so the two agree on
flags and num_mappings exactly and on rms / max_dist to rounding."""
import ctypes as C
import itertools
import json

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

MATCHED, COMPOSITION, DEGENERATE, SEARCH_LIMIT, TOO_LARGE = 1, 2, 4, 8, 16
MAX_ATOMS, BAND_CAP, MAX_STEPS, LLL_ITERS, NIGGLI_ITERS = 256, 128, 255, 1000, 100
_IMAGES = np.array(list(itertools.product((-1, 0, 1), repeat=3)), dtype=np.float64)


def lll_reduce(B, delta=0.75):
    """pymatgen Lattice._calculate_lll on the rows of B: (reduced rows, integer map with reduced = map @ B, converged)."""
    a = np.array(B, dtype=np.float64).T.copy()
    b, u, m = np.zeros((3, 3)), np.zeros((3, 3)), np.zeros(3)
    b[:, 0] = a[:, 0]
    m[0] = b[:, 0] @ b[:, 0]
    for i in range(1, 3):
        u[i, :i] = (a[:, i] @ b[:, :i]) / m[:i]
        b[:, i] = a[:, i] - b[:, :i] @ u[i, :i]
        m[i] = b[:, i] @ b[:, i]
    k, mapping, it = 2, np.eye(3), 0
    while k <= 3:
        it += 1
        if it > LLL_ITERS:
            return a.T, mapping.T, False
        for i in range(k - 1, 0, -1):
            q = np.round(u[k - 1, i - 1])
            if q != 0:
                a[:, k - 1] -= q * a[:, i - 1]
                mapping[:, k - 1] -= q * mapping[:, i - 1]
                u[k - 1, :i] -= q * np.append(u[i - 1, :i - 1], 1.0)
        if b[:, k - 1] @ b[:, k - 1] >= (delta - abs(u[k - 1, k - 2]) ** 2) * (b[:, k - 2] @ b[:, k - 2]):
            k += 1
        else:
            a[:, [k - 2, k - 1]] = a[:, [k - 1, k - 2]]
            mapping[:, [k - 2, k - 1]] = mapping[:, [k - 1, k - 2]]
            for s in range(k - 1, k + 1):
                u[s - 1, :s - 1] = (a[:, s - 1] @ b[:, :s - 1]) / m[:s - 1]
                b[:, s - 1] = a[:, s - 1] - b[:, :s - 1] @ u[s - 1, :s - 1]
                m[s - 1] = b[:, s - 1] @ b[:, s - 1]
            if k > 2:
                k -= 1
            else:
                u[k:3, k - 2:k] = (a[:, k:3].T @ b[:, k - 2:k]) / m[k - 2:k]
    return a.T, mapping.T, True


def g6(B):
    """(A, B, C, xi, eta, zeta) = (a.a, b.b, c.c, 2 b.c, 2 a.c, 2 a.b) of the rows of B."""
    G = B @ B.T
    return np.array([G[0, 0], G[1, 1], G[2, 2], 2 * G[1, 2], 2 * G[0, 2], 2 * G[0, 1]])


def niggli_reduce(B, tol=1e-5):
    """Krivy-Gruber with pymatgen's epsilon e = tol * V^(1/3), on the LLL-reduced basis (as pymatgen starts), applied
    to the basis rows so that the integer transform is kept: (Niggli rows, integer C with rows = C @ B, converged)."""
    e = tol * abs(np.linalg.det(B)) ** (1.0 / 3.0)
    b, C, ok = lll_reduce(B)
    if not ok:
        return b, C, False
    for _ in range(NIGGLI_ITERS):
        A, Bb, Cc, E, N, Y = g6(b)
        if A > Bb + e or (abs(A - Bb) < e and abs(E) > abs(N) + e):                    # A1
            b, C = -b[[1, 0, 2]], -C[[1, 0, 2]]
            A, Bb, Cc, E, N, Y = g6(b)
        if Bb > Cc + e or (abs(Bb - Cc) < e and abs(N) > abs(Y) + e):                  # A2
            b, C = -b[[0, 2, 1]], -C[[0, 2, 1]]
            continue
        l = 0 if abs(E) < e else np.sign(E)
        m = 0 if abs(N) < e else np.sign(N)
        n = 0 if abs(Y) < e else np.sign(Y)
        if l * m * n == 1:                                                              # A3
            d = np.array([-1 if l == -1 else 1, -1 if m == -1 else 1, -1 if n == -1 else 1], np.float64)
        else:                                                                           # A4
            d = np.array([-1 if l == 1 else 1, -1 if m == 1 else 1, -1 if n == 1 else 1], np.float64)
            if d.prod() == -1:
                if n == 0:
                    d[2] = -1
                elif m == 0:
                    d[1] = -1
                elif l == 0:
                    d[0] = -1
        b, C = b * d[:, None], C * d[:, None]
        A, Bb, Cc, E, N, Y = g6(b)
        if abs(E) > Bb + e or (abs(E - Bb) < e and 2 * N < Y - e) or (abs(E + Bb) < e and Y < -e):   # A5
            s = np.sign(E)
            b[2], C[2] = b[2] - s * b[1], C[2] - s * C[1]
            continue
        if abs(N) > A + e or (abs(A - N) < e and 2 * E < Y - e) or (abs(A + N) < e and Y < -e):      # A6
            s = np.sign(N)
            b[2], C[2] = b[2] - s * b[0], C[2] - s * C[0]
            continue
        if abs(Y) > A + e or (abs(A - Y) < e and 2 * E < N - e) or (abs(A + Y) < e and N < -e):      # A7
            s = np.sign(Y)
            b[1], C[1] = b[1] - s * b[0], C[1] - s * C[0]
            continue
        S = E + N + Y + A + Bb
        if S < -e or (abs(S) < e and e < Y + (A + N) * 2):                                          # A8
            b[2], C[2] = b[0] + b[1] + b[2], C[0] + C[1] + C[2]
            continue
        return b, C, True
    return b, C, False


def int_inv(S):
    return np.round(np.linalg.inv(S))


def wrap(f):
    return f - np.floor(f)


def params(M):
    """Lengths and angles (degrees, pymatgen's abs_cap + arccos) of the rows of M."""
    ln = np.sqrt((M * M).sum(1))
    ang = [np.arccos(np.clip(M[(d + 1) % 3] @ M[(d + 2) % 3] / (ln[(d + 1) % 3] * ln[(d + 2) % 3]), -1, 1))
           * 180.0 / np.pi for d in range(3)]
    return np.concatenate([ln, ang])


def from_params(p):
    """pymatgen Lattice.from_parameters (vesta=False)."""
    a, b, c = p[:3]
    al, be, ga = np.radians(p[3:])
    val = np.clip((np.cos(al) * np.cos(be) - np.cos(ga)) / (np.sin(al) * np.sin(be)), -1, 1)
    gs = np.arccos(val)
    return np.array([[a * np.sin(be), 0.0, a * np.cos(be)],
                     [-b * np.sin(al) * np.cos(gs), b * np.sin(al) * np.sin(gs), b * np.cos(al)],
                     [0.0, 0.0, c]])


def _recip(A):
    return np.sqrt((np.linalg.inv(A) ** 2).sum(0))      # |columns of A^-1|


def _result(flags, rms=np.nan, max_dist=np.nan, num_mappings=0):
    return dict(rms=rms, max_dist=max_dist, num_mappings=num_mappings, flags=flags)


def match_pair(f1, L1, z1, f2, L2, z2, stol=0.5, ltol=0.3, angle_tol=10.0):
    """rms, max_dist, num_mappings and flags of generated crystal (f1, L1, z1) against source (f2, L2, z2)."""
    f1, f2 = np.asarray(f1, np.float64).reshape(-1, 3), np.asarray(f2, np.float64).reshape(-1, 3)
    z1, z2 = np.asarray(z1, np.int64).reshape(-1), np.asarray(z2, np.int64).reshape(-1)
    o1, o2 = np.argsort(z1, kind="stable"), np.argsort(z2, kind="stable")
    f1, z1, f2, z2 = f1[o1], z1[o1], f2[o2], z2[o2]
    n = len(z1)
    if len(z2) != n or np.any(z1 != z2):
        return _result(COMPOSITION)
    if n > MAX_ATOMS:
        return _result(TOO_LARGE)
    L1, L2 = np.asarray(L1, np.float64), np.asarray(L2, np.float64)
    if n == 0 or not (np.isfinite(L1).all() and np.isfinite(L2).all() and np.isfinite(f1).all()
                      and np.isfinite(f2).all()):
        return _result(DEGENERATE)
    if not (abs(np.linalg.det(L1)) >= 0.1 and abs(np.linalg.det(L2)) >= 0.1):
        return _result(DEGENERATE)
    N1, C1, ok1 = niggli_reduce(L1)
    N2, C2, ok2 = niggli_reduce(L2)
    if not (ok1 and ok2):
        return _result(DEGENERATE)
    f1n, f2n = wrap(f1 @ int_inv(C1)), wrap(f2 @ int_inv(C2))
    ratio = (abs(np.linalg.det(N2)) / abs(np.linalg.det(N1))) ** (1.0 / 6.0)
    L1s, L2s = N1 * ratio, N2 / ratio
    p2 = params(L2s)
    rmax = p2[:3].max() * (1 + ltol)
    K = np.floor(rmax * _recip(L1s))
    if not np.all(K <= MAX_STEPS):
        return _result(SEARCH_LIMIT)
    grid = np.array(list(itertools.product(*[np.arange(-k, k + 1) for k in K])), dtype=np.float64)
    v = grid @ L1s
    d = np.sqrt((v * v).sum(1))
    bands = []
    for l in p2[:3]:
        q = d / l
        sel = np.nonzero((q < 1 + ltol) & (q > 1 / (1 + ltol)))[0]
        if len(sel) > BAND_CAP:
            return _result(SEARCH_LIMIT)
        bands.append(sel)

    def within(i, j, target):
        x = np.clip((v[i] @ v[j].T) / d[i][:, None] / d[j][None, :], -1, 1)
        return np.abs(np.arccos(x) * 180.0 / np.pi - target) < angle_tol

    A, B, C = bands
    alpha, beta, gamma = within(B, C, p2[3]), within(A, C, p2[4]), within(A, B, p2[5])
    blocks = np.concatenate([[0], np.nonzero(np.diff(z2))[0] + 1, [n]])
    sizes = np.diff(blocks)
    rare = int(np.argmin(sizes))                      # first of the rarest = smallest Z among ties
    anchor, t_sites = blocks[rare], np.arange(blocks[rare], blocks[rare + 1])
    same = z1[None, :] == z2[:, None]
    best, num_mappings = None, 0
    for i in range(len(A)):
        for j in range(len(B)):
            if not gamma[i, j]:
                continue
            for k in range(len(C)):
                if not (alpha[j, k] and beta[i, k]):
                    continue
                S = grid[[A[i], B[j], C[k]]]
                if abs(round(np.linalg.det(S))) != 1:
                    continue
                num_mappings += 1
                cand = _mapping(S, v[[A[i], B[j], C[k]]], f1n, f2n, p2, n, stol, blocks, anchor, t_sites, same)
                if cand is not None and (best is None or cand[0] < best[0]):
                    best = cand
    if best is None:
        return _result(0, num_mappings=num_mappings)
    return _result(MATCHED if best[0] < stol else 0, best[0], best[1], num_mappings)


def _mapping(S, M, f1n, f2n, p2, n, stol, blocks, anchor, t_sites, same):
    """Best (rms, max_dist) over the translations of one lattice mapping, or None."""
    fc1 = wrap(f1n @ int_inv(S))
    avg = from_params((params(M) + p2) / 2)
    norm = (n / abs(np.linalg.det(avg))) ** (1.0 / 3.0)
    frac_tol = 2 * stol * _recip(avg) / norm
    Bl, Mp, _ = lll_reduce(avg)
    lll_tol = 2 * stol * _recip(Bl) / norm
    Mpinv = int_inv(Mp)
    lf1 = wrap(fc1 @ Mpinv)
    im = _IMAGES @ Bl
    best = None
    for t in fc1[t_sites] - f2n[anchor]:
        dd = (f2n + t)[:, None, :] - fc1[None, :, :]                         # prefilter: is_coord_subset_pbc
        if not np.all(np.any(np.all(np.abs(dd - np.round(dd)) <= frac_tol, axis=-1) & same, axis=1)):
            continue
        lf2 = wrap((f2n + t) @ Mpinv)
        vecs = np.empty((n, 3))
        feasible = True
        for b0, b1 in zip(blocks[:-1], blocks[1:]):
            D = lf1[None, b0:b1] - lf2[b0:b1, None]                          # rows s2, columns s1
            adm = np.all(np.abs(D - np.round(D)) <= lll_tol, axis=-1)
            cart = (D @ Bl)[:, :, None, :] + im[None, None]
            d2 = (cart * cart).sum(-1)
            kbest = np.argmin(d2, axis=-1)
            cost = np.where(adm, np.take_along_axis(d2, kbest[..., None], -1)[..., 0], np.inf)
            try:
                rows, cols = linear_sum_assignment(cost)
            except ValueError:                                               # no complete matching
                feasible = False
                break
            vecs[b0 + rows] = cart[rows, cols, kbest[rows, cols]]
        if not feasible:
            continue
        dist = np.sqrt(((vecs - vecs.mean(0)) ** 2).sum(1)) * norm
        rms = np.linalg.norm(dist) / np.sqrt(n)
        if best is None or rms < best[0]:
            best = (rms, dist.max())
    return best


def match_pairs(gen, ref, **kw):
    """match_pair over two (frac, lattice, z, num_atoms) tuples; arrays rms, max_dist, num_mappings, flags."""
    o1, o2 = np.concatenate([[0], np.cumsum(gen[3])]), np.concatenate([[0], np.cumsum(ref[3])])
    out = [match_pair(gen[0][o1[g]:o1[g + 1]], gen[1][g], gen[2][o1[g]:o1[g + 1]],
                      ref[0][o2[g]:o2[g + 1]], ref[1][g], ref[2][o2[g]:o2[g + 1]], **kw) for g in range(len(gen[3]))]
    return {k: np.array([o[k] for o in out]) for k in ("rms", "max_dist", "num_mappings", "flags")}


# ---- helpers shared with the GPU tests ------------------------------------------------------------------------------
def random_unimodular(rng, steps=3):
    U = np.eye(3)
    for _ in range(steps):
        E = np.eye(3)
        i, j = rng.choice(3, 2, replace=False)
        E[i, j] = rng.integers(-2, 3)
        U = E @ U
    return U * rng.choice([-1.0, 1.0])


def random_rotation(rng):
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    return q * np.sign(np.diag(r))


def transformed_copy(f, L, z, rng, sigma=0.0, scale=True):
    """The same crystal re-based by a random unimodular matrix, rotated, translated, permuted and (scale) volume-scaled
    by up to +-10 %, its atoms displaced by Gaussian Cartesian noise of sigma * (V / n)^(1/3) per axis."""
    n = len(z)
    U = random_unimodular(rng)
    s = (1 + rng.uniform(-0.1, 0.1)) ** (1 / 3) if scale else 1.0
    L2 = U @ L @ random_rotation(rng) * s
    f2 = f @ np.linalg.inv(U) + rng.random(3)
    f2 = f2 + rng.standard_normal((n, 3)) * sigma * (abs(np.linalg.det(L2)) / n) ** (1 / 3) @ np.linalg.inv(L2)
    perm = rng.permutation(n)
    return wrap(f2)[perm], L2, np.asarray(z)[perm]


def random_cell(rng, n):
    a = np.cbrt(18.05 * n)
    L = np.diag(a * (1 + 0.1 * rng.standard_normal(3)))
    L[1, 0], L[2, :2] = a * 0.2 * rng.standard_normal(), a * 0.2 * rng.standard_normal(2)
    return L


# ---- CPU ------------------------------------------------------------------------------------------------------------
def _cell_from_g6(v):
    A, B, Cc, xi, eta, zeta = v
    return np.linalg.cholesky(np.array([[A, zeta / 2, eta / 2], [zeta / 2, B, xi / 2], [eta / 2, xi / 2, Cc]]))


def _assert_niggli_conditions(v, tol):
    A, B, Cc, xi, eta, zeta = v
    assert A <= B + tol and B <= Cc + tol
    assert abs(xi) <= B + tol and abs(eta) <= A + tol and abs(zeta) <= A + tol
    assert (xi > 0 and eta > 0 and zeta > 0) or (xi <= tol and eta <= tol and zeta <= tol)
    assert xi + eta + zeta + A + B >= -tol


def test_niggli_krivy_gruber_example():
    L = _cell_from_g6((9, 27, 4, -5, -4, -22))
    b, T, ok = niggli_reduce(L)
    assert ok
    np.testing.assert_allclose(g6(b), [4, 9, 9, 9, 3, 4], atol=1e-12)
    np.testing.assert_allclose(np.linalg.det(b @ b.T), 213.75, rtol=1e-12)
    np.testing.assert_allclose(np.linalg.det(L @ L.T), 213.75, rtol=1e-12)
    np.testing.assert_allclose(T @ L, b, atol=1e-12)                # the integer transform is kept
    assert np.array_equal(T, np.round(T)) and abs(round(np.linalg.det(T))) == 1


def test_niggli_is_invariant_under_unimodular_transforms():
    rng = np.random.default_rng(0)
    for _ in range(200):
        L = random_cell(rng, int(rng.integers(1, 30)))
        ref, _, ok = niggli_reduce(L)
        assert ok
        _assert_niggli_conditions(g6(ref), 1e-9 * g6(ref)[:3].max())
        for _ in range(3):
            U = random_unimodular(rng, steps=int(rng.integers(1, 6)))
            b, T, ok = niggli_reduce(U @ L @ random_rotation(rng))
            assert ok
            np.testing.assert_allclose(g6(b), g6(ref), rtol=0, atol=1e-9)


def test_exact_copies_match():
    rng = np.random.default_rng(1)
    for _ in range(30):
        n = int(rng.integers(1, 13))
        f, L, z = rng.random((n, 3)), random_cell(rng, n), rng.integers(1, 5, n)
        f2, L2, z2 = transformed_copy(f, L, z, rng)
        r = match_pair(f2, L2, z2, f, L, z)
        assert r["flags"] == MATCHED and r["rms"] <= 1e-10 and r["max_dist"] <= 1e-10 and r["num_mappings"] >= 1


def test_zero_mean_displacements_give_the_analytic_rms():
    rng = np.random.default_rng(2)
    for _ in range(20):
        n = int(rng.integers(2, 13))
        f, L, z = rng.random((n, 3)), random_cell(rng, n), rng.integers(1, 4, n)
        d = rng.standard_normal((n, 3)) * 0.01 * (abs(np.linalg.det(L)) / n) ** (1 / 3)
        d -= d.mean(0)
        r = match_pair(wrap(f + d @ np.linalg.inv(L)), L, z, f, L, z)
        expect = np.sqrt((d * d).sum(1).mean()) * (n / abs(np.linalg.det(L))) ** (1 / 3)
        assert r["flags"] == MATCHED
        assert abs(r["rms"] - expect) <= 1e-10, (r, expect)
        assert abs(r["max_dist"] - np.sqrt((d * d).sum(1)).max() * (n / abs(np.linalg.det(L))) ** (1 / 3)) <= 1e-10


def test_swapped_or_changed_elements_do_not_match():
    # an A layer at z ~ 0 and a B layer at z ~ 0.5 of a long cell: swapping an A and a B atom moves each by c / 2
    L = np.array([[3.0, 0, 0], [0.2, 3.1, 0], [0.3, -0.2, 12.0]])
    f = np.array([[0.0, 0.0, 0.0], [0.5, 0.5, 0.02], [0.0, 0.5, 0.5], [0.5, 0.0, 0.53]])
    z = np.array([8, 8, 26, 26])
    assert match_pair(f, L, z, f, L, z)["flags"] == MATCHED
    r = match_pair(f[[2, 1, 0, 3]], L, z, f, L, z)
    assert r["flags"] == 0 and r["num_mappings"] > 0 and not r["rms"] < 0.5     # no translation passes the prefilter
    assert match_pair(f, L, [8, 8, 26, 27], f, L, z)["flags"] == COMPOSITION
    assert match_pair(f[:3], L, z[:3], f, L, z)["flags"] == COMPOSITION


def test_match_summary_counts():
    from arreau_b200.inference.crystal_metrics import CrystalMetrics
    from arreau_b200.inference.structure_match import StructureMatch, match_summary
    flags = np.array([1, 1, 0, 2, 8, 4, 16, 1], np.int32)
    m = StructureMatch(matched=(flags & 1) != 0, rms=np.array([0.1, 0.3, 0.6, np.nan, np.nan, np.nan, np.nan, 0.2]),
                       max_dist=np.zeros(8), num_mappings=np.ones(8, np.int32), flags=flags)
    gen = CrystalMetrics(num_atoms=np.ones(8, np.int64), volume=np.ones(8), min_dist=np.ones(8), density=np.ones(8),
                         num_elements=np.ones(8, np.int32), flags=np.array([1, 1, 1, 1, 1, 1, 1, 0], np.int32))
    s = match_summary(m, gen)
    assert s["num_pairs"] == 8 and s["num_matched"] == 2 and s["match_rate"] == 0.25
    assert abs(s["mean_rms"] - 0.2) < 1e-15
    assert (s["num_composition_mismatch"], s["num_match_search_limit"], s["num_match_degenerate"],
            s["num_too_large"]) == (1, 1, 1, 1)
    json.dumps(s)


def test_match_entry_point_argument_validation():
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p)
    args = lambda **kw: [kw.get(k, v) for k, v in (  # noqa: E731
        ("f1", p), ("l1", p), ("z1", p), ("o1", p), ("f2", p), ("l2", p), ("z2", p), ("o2", p), ("n1", 4), ("n2", 4),
        ("g", 1), ("stol", 0.5), ("ltol", 0.3), ("atol", 10.0), ("rms", p), ("md", p), ("nm", p), ("fl", p),
        ("stream", None))]
    assert lib.arreau_structure_match(*args(g=0, f1=None, l1=None, rms=None)) == 0
    for k in ("l1", "o1", "l2", "o2", "rms", "md", "nm", "fl", "f1", "z1", "f2", "z2"):
        assert lib.arreau_structure_match(*args(**{k: None})) == -4, k
    assert lib.arreau_structure_match(*args(n1=0, f1=None, z1=None, g=-1)) == -1
    for kw in (dict(g=-1), dict(n1=-4), dict(n2=-4), dict(stol=0.0), dict(ltol=-0.3), dict(atol=float("nan")),
               dict(stol=float("inf"))):
        assert lib.arreau_structure_match(*args(**kw)) == -1, kw


def _cli_files(tmp_path, source_index=True, index=None):
    from arreau_b200.diffusion.diffusion_loss import SampleResult
    from arreau_b200.diffusion.lattice_dataset import save_dataset_npz
    from arreau_b200.inference.process_generated_crystals import save_sample_results_to_hdf5
    rng = np.random.default_rng(3)
    zs = [rng.integers(1, 9, 3) for _ in range(4)]
    lats = np.stack([random_cell(rng, 3) for _ in range(4)])
    fr = [rng.random((3, 3)) for _ in range(4)]
    data = save_dataset_npz(str(tmp_path / "data"), zs, lats, fr)
    idx = np.array([2, 0, 3] if index is None else index, np.int64)
    src = idx % 4                        # the crystals written; idx itself may point outside the data set
    res = SampleResult(frac_x=np.concatenate([fr[i] for i in src]), lattice=lats[src],
                       atomic_numbers=np.concatenate([zs[i] for i in src]), num_atoms=np.full(len(idx), 3),
                       idx_start=np.arange(len(idx)) * 3)
    out = save_sample_results_to_hdf5(res, str(tmp_path / "crystals.npz"), {"source_index": idx} if source_index else None)
    return out, data


def test_match_cli_refusals(tmp_path, capsys):
    from arreau_b200.inference import crystal_metrics
    from arreau_b200.inference.process_generated_crystals import load_extra_arrays
    out, data = _cli_files(tmp_path)
    assert np.array_equal(load_extra_arrays(out, ("source_index", "missing"))["source_index"], [2, 0, 3])
    assert list(load_extra_arrays(out, ("missing",))) == []
    cases = [([out, "--match"], "--match needs --reference")]
    cases.append(([_cli_files(tmp_path / "a", source_index=False)[0], "--reference", data, "--match"], "no source_index"))
    cases.append(([_cli_files(tmp_path / "b", index=[1, 4])[0], "--reference", data, "--match"], "outside"))
    cases.append(([_cli_files(tmp_path / "c", index=[-1, 0])[0], "--reference", data, "--match"], "outside"))
    for argv, what in cases:
        with pytest.raises(SystemExit):
            crystal_metrics.main(argv)
        assert what in capsys.readouterr().err, argv
