"""
The exact fixed-point Gram product of the Gaussian step's constant-weight SYRK (DESIGN §2), modelled in NumPy and pinned on the CPU.

    A = rint(Kuf * 2^52 / v)              0 <= A < 2^53, exact in a double (v = the kernel variance; Kuf may exceed v by rounding)
    r_i = A mod p_i  (symmetric range)    16 pairwise coprime moduli, int8 planes
    C_i = R_i R_i^T  (int32, exact)       < 2^31 for fewer than 2^17 points per slab
    B' = CRT(C_i mod p_i)                 Garner digits + Horner, symmetric range: exact while |B'| < P / 2
    B += alpha v^2 2^-104 double(B')      one rounding of the exact integer
"""
import numpy as np
import pytest
import scipy.linalg as sla

from tests.int8_gram_ref import GRID, MAX_POINTS, MODULI, P, crt, exact_gram, grid, modular_gram, residues, to_double

def emulated_gram(K, v, alpha=1.0):
    return to_double(crt(modular_gram(residues(grid(K, v)))), v, alpha)


def test_moduli_are_pairwise_coprime_and_cover_the_slab_bound():
    from math import gcd
    for i, p in enumerate(MODULI):
        for q in MODULI[i + 1:]:
            assert gcd(p, q) == 1
    # |B'| <= n (2^53 - 1)^2 < n 2^106 < P / 2 for every slab width the path takes
    assert MAX_POINTS * (2 ** 53 - 1) ** 2 < P // 2
    assert MAX_POINTS * 128 * 128 < 2 ** 31 <= (MAX_POINTS + 128) * 128 * 128
    # the grid keeps one bit of headroom above v: Kuf up to v (1 + 2^-52 * 2^k) still rounds below 2^53
    v = 1.7
    A = grid(np.array([0.0, v, np.nextafter(v, 2 * v), v * (1 + 1.5e-14), v * 1.999999]), v)
    assert A.max() < 2 ** 53 and np.all(A == np.floor(A))


def test_residues_reconstruct_every_grid_integer():
    rng = np.random.default_rng(0)
    A = np.concatenate([[0, 1, 2 ** 52, 2 ** 53 - 1, 2 ** 52 + 64], rng.integers(0, 2 ** 53, 200)]).astype(np.float64)[None, :]
    R = residues(A)
    for p, r in zip(MODULI, R):
        assert r.min() >= -(p // 2) and r.max() <= (p - 1) // 2
    back = crt([(r.astype(np.int64) % p) for p, r in zip(MODULI, R)])
    assert all(int(b) == int(a) for a, b in zip(A[0], back[0]))


def test_gram_is_the_exact_integer_rounded_once():
    rng = np.random.default_rng(1)
    v = 0.6
    K = v * rng.uniform(0.0, 1.0, size=(6, 2048))
    K[0, :5] = [0.0, v, np.nextafter(v, 1.0), v * (1 + 1.4e-14), 0.0]   # zero, exactly the variance, above it by rounding
    K[1, :] = 0.0
    K[2, 7] = np.nan                                                       # non-finite maps to 0 (the point kernel flags the step)
    A = grid(K, v)
    assert A.max() < 2 ** 53
    B_int = crt(modular_gram(residues(A)))
    assert np.array_equal(B_int, exact_gram(A))
    want = to_double(exact_gram(A), v, alpha=-3.5)
    got = emulated_gram(K, v, alpha=-3.5)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))


def test_widest_slab_at_the_largest_grid_values():
    # every entry at the top of the grid and at the variance: the int32 sums stay exact just below 2^17 points
    n = MAX_POINTS
    A = np.full((3, n), 2.0 ** 53 - 1)
    A[1] = 2.0 ** 52
    A[2, ::2] = 0.0
    R = residues(A)
    C = modular_gram(R)
    B_int = crt(C)
    assert np.array_equal(B_int, exact_gram(A))
    assert int(B_int[0, 0]) == n * (2 ** 53 - 1) ** 2


def _se(X, Z, var, ls):
    d2 = ((X[:, None, :] - Z[None, :, :]) ** 2).sum(-1) / ls ** 2
    return var * np.exp(-0.5 * d2)


def test_grid_error_is_below_fp64_reordering_in_G2():
    # cfg3's shape at reduced size: Z = X[:M], jitter 1e-9.  The grid's perturbation of B, exactly:
    #   K = A 2^-52 v + E  =>  K K^T - v^2 2^-104 A A^T = v 2^-52 (A E^T + E A^T) + E E^T   (E = K - A 2^-52 v exactly)
    rng = np.random.default_rng(3)
    N, M, D, v = 8192, 128, 16, 1.0
    X = rng.standard_normal((N, D))
    Z = X[:M]
    Kuf = _se(Z, X, v, 4.0)
    K9 = _se(Z, Z, v, 4.0) + 1e-9 * np.eye(M)
    A = grid(Kuf, v)
    Ag = A * (v / GRID)
    E = Kuf - Ag
    dB_grid = Ag @ E.T + E @ Ag.T + E @ E.T
    B_blas = Kuf @ Kuf.T
    B_pieces = sum(Kuf[:, i:i + 4096] @ Kuf[:, i:i + 4096].T for i in range(0, N, 4096))
    dB_order = B_blas - B_pieces
    c = sla.cho_factor(K9)
    g2 = lambda dB: sla.cho_solve(c, sla.cho_solve(c, dB).T)   # K9^-1 dB K9^-1
    G2 = g2(B_blas)
    e_grid = np.abs(g2(dB_grid)).max() / np.abs(G2).max()
    e_order = np.abs(g2(dB_order)).max() / np.abs(G2).max()
    assert np.abs(dB_grid).max() < np.abs(dB_order).max()
    assert e_grid * 10 < e_order, (e_grid, e_order)
