"""The per-crystal keyed draws (arreau_eval_noise, arreau_sample_init_keyed, arreau_sample_noise_keyed) against a numpy
Philox4x32-10 with the same counter words, tag words, u01 and Box-Muller, so that a changed counter, tag or
transform fails here and not only as a shift in moments.

Timesteps, uniforms and angles are compared bit for bit.  The normals go through the device's log and sincospi, which
are not correctly rounded, so they are compared within 4 ulp of an extended-precision reference."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

M32 = np.uint64(0xFFFFFFFF)
SEED = 0x9E3779B97F4A7C15
IDS = np.array([0, 5, (1 << 40) + 3, (1 << 63) - 1], dtype=np.int64)   # ids that need all 64 counter bits
COUNTS = np.array([1, 4, 3, 2])
Z = 7                                                                   # odd: the last uniform pair is cut in half


def philox4x32_10(seed, ctr_lo, ctr_hi, tag):
    """Random123's Philox4x32-10 on counter {ctr_lo (64 bits), ctr_hi, tag} and key seed; arrays broadcast."""
    ctr_lo = np.asarray(ctr_lo).astype(np.uint64)
    c = [ctr_lo & M32, ctr_lo >> np.uint64(32), np.asarray(ctr_hi).astype(np.uint64) & M32,
         np.asarray(tag).astype(np.uint64) & M32]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def u01(a, b):
    v = ((a << np.uint64(21)) ^ (b >> np.uint64(11))) & np.uint64((1 << 53) - 1)
    return v.astype(np.float64) * 2.0 ** -53


PI = np.longdouble("3.14159265358979323846264338327950288")


def box_muller(r):
    """Both normals of one Philox output in extended precision: sqrt(-2 log u1) (cos, sin)(2 pi u2)."""
    u1, x = 1.0 - u01(r[0], r[1]), 2.0 * u01(r[2], r[3])     # both exact
    k = np.rint(2.0 * x).astype(np.int64)                     # x = k / 2 + h exactly, |h| <= 1/4
    h = (x - 0.5 * k).astype(np.longdouble)
    s, c = np.sin(PI * h), np.cos(PI * h)
    q = k % 4
    sin = np.select([q == 0, q == 1, q == 2], [s, c, -s], -c)
    cos = np.select([q == 0, q == 1, q == 2], [c, -s, -c], s)
    rad = np.sqrt(-2.0 * np.log(u1.astype(np.longdouble)))
    return rad * cos, rad * sin


def reference(Zr, cell, len_tag, len_ctr0, frac_tag, type_tag):
    """Per-crystal uniform, lengths [G,3] and per-atom normals [N,3] (extended precision), uniforms [N,Z] (exact)."""
    g_of_atom = np.repeat(np.arange(len(IDS)), COUNTS)
    a = np.concatenate([np.arange(n) for n in COUNTS]).astype(np.uint64)
    ids, atom_ids = IDS.view(np.uint64), IDS.view(np.uint64)[g_of_atom]
    cu = u01(*philox4x32_10(SEED, ids, 0, cell)[:2]) if cell is not None else None
    l0, l1 = box_muller(philox4x32_10(SEED, ids, len_ctr0, len_tag))
    l2, _ = box_muller(philox4x32_10(SEED, ids, len_ctr0 + 1, len_tag))
    f0, f1 = box_muller(philox4x32_10(SEED, atom_ids, 2 * a, frac_tag))
    f2, _ = box_muller(philox4x32_10(SEED, atom_ids, 2 * a + np.uint64(1), frac_tag))
    H = (Zr + 1) // 2
    u = np.zeros((len(a), 2 * H))
    for k in range(H):
        r = philox4x32_10(SEED, atom_ids, a * np.uint64(H) + np.uint64(k), type_tag)
        u[:, 2 * k], u[:, 2 * k + 1] = u01(r[0], r[1]), u01(r[2], r[3])
    return cu, np.stack([l0, l1, l2], 1), np.stack([f0, f1, f2], 1), u[:, :Zr]


def assert_ulps(dev, ref, n=4):
    ref64 = ref.astype(np.float64)
    err = np.abs(dev.astype(np.longdouble) - ref)
    assert np.all(err <= n * np.spacing(np.abs(ref64)).astype(np.longdouble)), np.max(err / np.spacing(np.abs(ref64)))


def test_philox_known_answers():
    """Random123's known-answer vectors for philox4x32_10 (all-zero and all-one counter and key)."""
    assert [int(x) for x in philox4x32_10(0, 0, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    ones = philox4x32_10((1 << 64) - 1, np.uint64((1 << 64) - 1), 0xFFFFFFFF, 0xFFFFFFFF)
    assert [int(x) for x in ones] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def _buffers(device):
    import torch
    off = torch.tensor(np.concatenate([[0], np.cumsum(COUNTS)]), dtype=torch.int32, device=device)
    coa = torch.tensor(np.repeat(np.arange(len(COUNTS)), COUNTS), dtype=torch.int32, device=device)
    ids = torch.tensor(IDS, device=device)
    nan = lambda *s: torch.full(s, float("nan"), dtype=torch.float64, device=device)  # noqa: E731
    return off, coa, ids, nan, torch.cuda.current_stream().cuda_stream


@pytest.mark.gpu
def test_eval_noise_matches_reference(device):
    import torch
    from arreau_b200 import _lib
    off, coa, ids, nan, s = _buffers(device)
    G, N, T = len(IDS), int(COUNTS.sum()), 1000
    t = torch.zeros(G, dtype=torch.int32, device=device)
    eps_x, u, eps_l = nan(N, 3), nan(N, Z), nan(G, 3)
    _lib.call("arreau_eval_noise", C.c_uint64(SEED), G, N, Z, T, ids.data_ptr(), off.data_ptr(), coa.data_ptr(),
              t.data_ptr(), eps_x.data_ptr(), u.data_ptr(), eps_l.data_ptr(), s)
    cu, lengths, frac, u_ref = reference(Z, 2, 3, 0, 4, 5)
    np.testing.assert_array_equal(t.cpu().numpy(), np.minimum(1 + (cu * T).astype(np.int64), T))
    assert u.cpu().numpy().tobytes() == u_ref.tobytes()
    assert_ulps(eps_l.cpu().numpy(), lengths)
    assert_ulps(eps_x.cpu().numpy(), frac)


@pytest.mark.gpu
def test_sample_init_keyed_matches_reference(device):
    from arreau_b200 import _lib
    off, coa, ids, nan, s = _buffers(device)
    G, N, scale = len(IDS), int(COUNTS.sum()), 0.7
    angles, lengths, frac = nan(G, 3), nan(G, 3), nan(N, 3)
    _lib.call("arreau_sample_init_keyed", C.c_uint64(SEED), G, N, ids.data_ptr(), off.data_ptr(), coa.data_ptr(), scale,
              angles.data_ptr(), lengths.data_ptr(), frac.data_ptr(), s)
    cu, len_ref, frac_ref, _ = reference(0, 6, 6, 1, 7, 0)
    # beta = 90 + 90 u, rounded once (the device contracts it into one fused multiply-add)
    beta = [float(90 + 90 * Fraction(float(x))) for x in cu]
    a = angles.cpu().numpy()
    assert a[:, 1].tobytes() == np.array(beta).tobytes() and np.all(a[:, [0, 2]] == 90.0)
    assert_ulps(lengths.cpu().numpy(), len_ref)
    assert_ulps(frac.cpu().numpy(), frac_ref * np.longdouble(scale))


@pytest.mark.gpu
@pytest.mark.parametrize("step", [0, 7, (1 << 28) - 1])
def test_sample_noise_keyed_matches_reference(device, step):
    from arreau_b200 import _lib
    off, coa, ids, nan, s = _buffers(device)
    G, N = len(IDS), int(COUNTS.sum())
    z_len, z_frac, u = nan(G, 3), nan(N, 3), nan(N, Z)
    _lib.call("arreau_sample_noise_keyed", C.c_uint64(SEED), step, G, N, Z, ids.data_ptr(), off.data_ptr(),
              coa.data_ptr(), z_len.data_ptr(), z_frac.data_ptr(), u.data_ptr(), s)
    hi = step << 4
    _, len_ref, frac_ref, u_ref = reference(Z, None, 8 | hi, 0, 9 | hi, 10 | hi)
    assert u.cpu().numpy().tobytes() == u_ref.tobytes()
    assert_ulps(z_len.cpu().numpy(), len_ref)
    assert_ulps(z_frac.cpu().numpy(), frac_ref)
