"""NumPy model of the INT8 contractions' slice splitting (tools/int8gemm/emulate_ozaki.py, csrc/gemm_int8.cu)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "int8gemm"))
import emulate_ozaki as oz  # noqa: E402


def _Y(rng, L, M):
    Y = rng.standard_normal((L, M)) * np.ldexp(1.0, rng.integers(-30, 31, L))[:, None] * np.ldexp(1.0, rng.integers(-30, 31, M))[None, :]
    Y[3, :] = 0.0
    Y[:, 5] = 0.0
    return Y


def test_exponents_bound_and_zero_lines():
    Y = _Y(np.random.default_rng(1), 40, 30)
    F, E, Z = oz.scale_Y(Y)
    assert np.all(np.abs(Z) < 1.0)
    assert F[3] == 0 and E[5] == 0 and np.all(Z[3, :] == 0) and np.all(Z[:, 5] == 0)
    # every nonzero column reaches [1/2, 1): the scale is tight
    nz = np.any(Z != 0, axis=0)
    assert np.all(np.max(np.abs(Z[:, nz]), axis=0) >= 0.5)
    assert np.array_equal(np.ldexp(np.ldexp(Z, F[:, None]), E[None, :]), Y)


def test_reconstruction_up_to_2_pow_minus_56():
    rng = np.random.default_rng(2)
    Z = rng.uniform(-1, 1, 20000) * (1 - 2.0 ** -53)
    Z[:4] = [0.0, 1 - 2.0 ** -53, -(1 - 2.0 ** -53), 2.0 ** -60]
    S = oz.split(Z)
    assert all(np.max(np.abs(s)) <= 127 for s in S)
    rec = sum(np.ldexp(s.astype(np.float64), -7 * (i + 1)) for i, s in enumerate(S))
    assert np.max(np.abs(Z - rec)) < 2.0 ** -56
    # slices share the sign of the value (truncation toward zero)
    assert all(np.all(s * np.sign(Z) >= 0) for s in S)


def test_overflow_bound_of_level_7():
    # level 7 sums the 8 products i + j = 7 of |S| <= 127; the kernel flushes every 16384 k
    per_k = 8 * 127 * 127
    assert per_k * 16384 < 2 ** 31 - 1
    assert (2 ** 31 - 1) // per_k == 16643
    # every slice at 127: the largest level sums reach the bound without wrapping in int64
    S = [np.full((16384, 1), 127, np.int64)] * 8
    lev7 = sum(S[i].T @ S[7 - i] for i in range(8))
    assert int(lev7[0, 0]) == per_k * 16384 < 2 ** 31


def test_combination_order_is_levels_7_to_0():
    rng = np.random.default_rng(3)
    levels = [rng.integers(-2 ** 30, 2 ** 30, 1000) for _ in range(8)]
    explicit = np.zeros(1000)
    for k in range(7, -1, -1):
        explicit = explicit + np.ldexp(levels[k].astype(np.float64), -7 * (k + 2))
    assert np.array_equal(oz.combine(levels), explicit)


def test_product_matches_float64():
    rng = np.random.default_rng(4)
    Y = _Y(rng, 300, 200)
    B = rng.standard_normal((300, 7)) * np.exp(rng.uniform(-6, 2, 7))[None, :]
    A = rng.standard_normal((200, 7))
    P, Q = oz.k1(Y, B), oz.k2(Y, A)
    assert oz.rel(P, Y.T @ B) < 1e-13
    assert oz.rel(Q, Y @ A) < 1e-13
    # integer-valued inputs are exact
    Yi = rng.integers(-1000, 1000, (300, 200)).astype(np.float64)
    Bi = rng.integers(-1000, 1000, (300, 7)).astype(np.float64)
    assert np.array_equal(oz.k1(Yi, Bi), Yi.T @ Bi)
