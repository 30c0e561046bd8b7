"""NumPy model of the INT8 contractions' signed radix-256 digits (tools/int8gemm/emulate_ozaki.py, csrc/gemm_int8.cu)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "int8gemm"))
import emulate_ozaki as oz  # noqa: E402

EDGE = 127.0 / 128.0


def _adversarial():
    """values |Z| <= 127/128 at the ends of the digit range, around the rounding of the last digit and near zero"""
    rng = np.random.default_rng(21)
    v = [0.0, EDGE, -EDGE, np.nextafter(EDGE, 0), -np.nextafter(EDGE, 0), 2.0 ** -60, -2.0 ** -60, 2.0 ** -56, 3 * 2.0 ** -57,
         -3 * 2.0 ** -57, 0.5, -0.5, 1.0 / 255, -128.0 / 255, 127.0 / 255]
    # every digit at its ends: -128 * sum 256^-i (inside the bound from the second digit on) and 127 * sum 256^-i
    for d in (-128, 127, -127):
        for top in range(1, 7):
            X = sum(d * 256 ** i for i in range(7 - top))
            v.append(float(X) * 2.0 ** -55)
    return np.concatenate([np.array(v), rng.uniform(-EDGE, EDGE, 20000)])


def test_digit_range_and_remainder():
    Z = _adversarial()
    X = np.rint(np.ldexp(Z, 55)).astype(np.int64)
    assert np.max(np.abs(X)) <= 127 * 2 ** 48
    D, rest = oz.digits_of(X)
    assert len(D) == 7 and not np.any(rest)
    lo, hi = min(int(d.min()) for d in D), max(int(d.max()) for d in D)
    assert lo == -128 and hi == 127
    # the digits are exactly the integer back
    assert np.array_equal(sum(d * 256 ** (6 - i) for i, d in enumerate(D)), X)
    # the ends of the integer range itself: -128 (2^56 - 1) / 255 .. 127 (2^56 - 1) / 255, and one past them is left over
    top = (2 ** 56 - 1) // 255
    for x, ok in ((-128 * top, True), (127 * top, True), (-128 * top - 1, False), (127 * top + 1, False)):
        D, rest = oz.digits_of(np.array([x]))
        assert (not np.any(rest)) == ok
        if ok:
            assert all(-128 <= int(d[0]) <= 127 for d in D)


def test_reconstruction_up_to_2_pow_minus_56():
    Z = _adversarial()
    D = oz.split_digits(Z)
    rec = sum(np.ldexp(d.astype(np.float64), -(7 + 8 * i)) for i, d in enumerate(D))
    assert np.max(np.abs(Z - rec)) <= 2.0 ** -56
    # rounding to nearest: the error is symmetric, not biased toward zero as truncation is
    err = (Z - rec)[-20000:]
    assert abs(np.mean(np.sign(err) * np.sign(Z[-20000:]))) < 0.05


def test_exponent_rule():
    rng = np.random.default_rng(22)
    L, M = 40, 30
    Y = rng.standard_normal((L, M)) * np.ldexp(1.0, rng.integers(-30, 31, L))[:, None] * np.ldexp(1.0, rng.integers(-30, 31, M))[None, :]
    Y[3, :] = 0.0
    Y[:, 5] = 0.0
    Y[1, :] = rng.standard_normal(M) * 2.0 ** -1060   # a subnormal row
    Y[1, 5] = 0.0
    F, E, Z = oz.scale_Y_digits(Y)
    assert np.all(np.abs(Z) <= EDGE)
    assert F[3] == 0 and E[5] == 0 and np.all(Z[3, :] == 0) and np.all(Z[:, 5] == 0)
    assert np.array_equal(np.ldexp(Z, F[:, None] + E[None, :]), Y)
    # the rule is tight: the exponent is the smallest with |column| <= (127/128) 2^E
    nz = np.any(Z != 0, axis=0)
    assert np.all(np.max(np.abs(Z[:, nz]), axis=0) > EDGE / 2)
    assert np.array_equal(oz.exponent_digits(np.array([0.0, EDGE, np.nextafter(EDGE, 1), 1.0, 0.5, -EDGE * 4])), [0, 0, 1, 1, 0, 2])
    # column maxima just above and just below 127/128 and +-(1 - 2^-53): above 127/128 the exponent grows by one and halves
    # the value, at or below it the value stays
    v = np.array([np.nextafter(EDGE, 1), np.nextafter(EDGE, 0), 1 - 2.0 ** -53, -(1 - 2.0 ** -53)])
    F2, E2, Z2 = oz.scale_Y_digits(np.ldexp(np.stack([v, v / 4]), 40))
    assert list(F2) == [40, 38] and list(E2) == [1, 0, 1, 1]
    assert list(Z2[0]) == [v[0] / 2, v[1], v[2] / 2, v[3] / 2]
    # the subnormal row is scaled up exactly and its digits reconstruct it
    assert np.all((Z[1] != 0) == (Y[1] != 0)) and not np.any(oz.digits_of(np.rint(np.ldexp(Z[1], 55)).astype(np.int64))[1])


def test_level_6_bound_at_16384_k():
    # level 6 sums the 7 products i + j = 6 of |digit| <= 128; the kernel flushes every 16384 k
    per_k = 7 * 128 * 128
    assert per_k == 114688 and per_k * 16384 < 2 ** 31 - 1
    assert (2 ** 31 - 1) // per_k == 18724
    D = [np.full((16384, 1), -128, np.int64)] * 7
    lev6 = sum(oz.slice_matmul(D[i], D[6 - i]) for i in range(7))
    assert int(lev6[0, 0]) == per_k * 16384 < 2 ** 31
    # the largest level 6 reachable under |Z| <= 127/128 (the top digit cannot be -128) stays below the bound
    X = sum(d * 256 ** (6 - i) for i, d in enumerate([126, 127, 127, 127, 127, 127, 124]))
    w = float(X) * 2.0 ** -55
    assert w <= EDGE and float(np.rint(np.ldexp(w, 55))) == X
    D = oz.split_digits(np.array([w]))
    assert [int(d[0]) for d in D] == [126, 127, 127, 127, 127, 127, 124]
    assert sum(int(D[i][0]) * int(D[6 - i][0]) for i in range(7)) >= 0.95 * per_k


def test_combination_order_is_levels_6_to_0():
    rng = np.random.default_rng(23)
    levels = [rng.integers(-2 ** 30, 2 ** 30, 1000) for _ in range(7)]
    explicit = np.zeros(1000)
    for k in range(6, -1, -1):
        explicit = explicit + np.ldexp(levels[k].astype(np.float64), -(8 * k + 14))
    assert np.array_equal(oz.combine_digits(levels), explicit)


def test_no_worse_than_7_bit_slices_on_main_inputs():
    for _, _, _, Y, B, A in oz.main_cases():
        refP = oz.k1(Y, B, ns_y=10, ns_b=10, cut=18)
        refQ = oz.k2(Y, A, ns_y=10, ns_b=10, cut=18)
        assert oz.rel(oz.k1_digits(Y, B), refP) <= oz.rel(oz.k1(Y, B), refP)
        assert oz.rel(oz.k2_digits(Y, A), refQ) <= oz.rel(oz.k2(Y, A), refQ)


def test_product_matches_float64_and_integers_are_exact():
    rng = np.random.default_rng(24)
    Y = rng.standard_normal((300, 200)) * np.ldexp(1.0, rng.integers(-30, 31, 300))[:, None]
    B = rng.standard_normal((300, 7)) * np.exp(rng.uniform(-6, 2, 7))[None, :]
    A = rng.standard_normal((200, 7))
    assert oz.rel(oz.k1_digits(Y, B), Y.T @ B) < 1e-13
    assert oz.rel(oz.k2_digits(Y, A), Y @ A) < 1e-13
    Yi = rng.integers(-1000, 1001, (300, 200)).astype(np.float64)
    Bi = rng.integers(-1000, 1001, (300, 7)).astype(np.float64)
    Ai = rng.integers(-1000, 1001, (200, 7)).astype(np.float64)
    assert np.array_equal(oz.k1_digits(Yi, Bi), Yi.T @ Bi)
    assert np.array_equal(oz.k2_digits(Yi, Ai), Yi @ Ai)
