"""The bit-exact host model of the INT8 contractions (tests/int8_model.py): agreement with the error-level model of
tools/int8gemm/emulate_ozaki.py, a componentwise error bound against the exactly rounded product, and the split plan."""
import os
import sys

import numpy as np
import pytest

from tests import int8_model as im

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "int8gemm"))
import emulate_ozaki as oz  # noqa: E402

U = 2.0 ** -53


@pytest.fixture(scope="module")
def lib():
    import vbmf_b200_loader
    vbmf_b200_loader.build()
    return vbmf_b200_loader.load()._lib.load()


def _inputs(rng, L, M, H, spread=30):
    Y = rng.standard_normal((L, M)) * np.ldexp(1.0, rng.integers(-spread, spread + 1, L))[:, None] \
        * np.ldexp(1.0, rng.integers(-spread, spread + 1, M))[None, :]
    if L > 2 and M > 2:            # an all-zero row and column next to data (at L or M <= 2 they would be most or all of Y)
        Y[L // 2, :] = 0.0
        Y[:, M // 3] = 0.0
    B = rng.standard_normal((L, H)) * np.ldexp(1.0, rng.integers(-20, 21, H))[None, :]
    A = rng.standard_normal((M, H)) * np.ldexp(1.0, rng.integers(-20, 21, H))[None, :]
    if H > 2:
        B[:, H // 2] = 0.0
    return Y, B, A


@pytest.mark.parametrize("L,M,H", [(129, 161, 7), (300, 200, 64), (17, 1, 3), (1, 40, 1)])
def test_single_split_matches_error_level_model(L, M, H):
    rng = np.random.default_rng(L * 7 + M + H)
    Y, B, A = _inputs(rng, L, M, H)
    assert np.any(Y) and np.any(B) and np.any(A)
    if L <= 2 or M <= 2:                                        # no zero line: every row and column carries data
        assert np.all(Y != 0)
    plan = (1, 32 * ((L + 31) // 32), 1, 32 * ((M + 31) // 32))
    assert np.array_equal(im.k1(Y, B, plan), oz.k1_digits(Y, B))
    # emulate_ozaki.k2_digits runs K1's scheme on Y' (frexp rule on Y's columns, 127/128 rule on its rows), while the
    # kernel's K2 keeps Y's own F and E: the same digits scheme with other exponents, so it agrees to rounding level only
    Q, Qoz = im.k2(Y, A, plan), oz.k2_digits(Y, A)
    assert np.max(np.abs(Q - Qoz)) <= 2.0 ** -50 * np.max(np.abs(Y) @ np.abs(A))


def _bound_k1(Y, B, plan, i, h, ref):
    """Componentwise bound of |model - exactly rounded product| for P[i, h].

    Every element is x = 2^(row exp + col exp) (z + r) with |z| <= 127/128 held by seven digits and |r| <= 2^-56.  Per term
    of the sum, with W = 2^(E_i + G_h), the scheme loses at most
        W (|r_y||z_b| + |z_y||r_b| + |r_y r_b|)   <= 2.01 W 2^-56   (representation)
      + W sum_{k=7..12} (13 - k) 128^2 2^-(14+8k) <= 6.03 W 2^-56   (the digit products i + j >= 7 that no level holds),
    so n terms lose at most 9 n W 2^-56.  The levels are exact integers.  Each later rounding (six fma of the combination,
    the ldexp, the add of each flush segment and of each slab, the eight subset adds of the wide sum) is at most u times a
    partial sum, and every partial sum is below 1.02 n W (sum of |digit| 2^-(7+8i) <= 1.004).  With R such roundings, and
    2^-1074 absolute each when the result is subnormal, plus half an ulp between the exact and the rounded reference:
        |model - ref| <= n W (9 2^-56 + 1.02 R u) + R 2^-1074 + u |ref|."""
    L = Y.shape[0]
    F, E = im.y_exponents(Y)
    G = im._masked_max(im.exp_digits(B) + F[:, None], B != 0, 0)
    S1, klen = plan[0], plan[1]
    nseg = sum(-(-(min(L, (s + 1) * klen) - s * klen) // im.SEG_K) for s in range(S1))
    R = 8 * nseg + S1 + 8
    W = np.ldexp(1.0, int(E[i] + G[h]))
    return L * W * (9 * 2.0 ** -56 + 1.02 * R * U) + R * 2.0 ** -1074 + U * abs(ref)


def _bound_k2(Y, A, plan, l, h, ref):
    """The same bound for Q[l, h]: W and n per split-K chunk, W_c = 2^(F_l + G_ch)."""
    M = Y.shape[1]
    F, E = im.y_exponents(Y)
    S, kchunk = plan[2], plan[3]
    tot, R = 0.0, S + 8
    for c in range(S):
        m0, m1 = c * kchunk, min(M, (c + 1) * kchunk)
        Gc = im._masked_max(im.exp_digits(A[m0:m1, h]) + E[m0:m1], A[m0:m1, h] != 0, 0)
        tot += (m1 - m0) * np.ldexp(1.0, int(F[l] + Gc))
        R += 8 * -(-(m1 - m0) // im.SEG_K)
    return tot * (9 * 2.0 ** -56 + 1.02 * R * U) + R * 2.0 ** -1074 + U * abs(ref)


@pytest.mark.parametrize("L,M,H,S1,kbs1,S2,kchunk", [
    (2000, 3001, 7, 2, 64, 6, 512),        # a few splits, ragged last ones
    (20000, 300, 5, 16, 80, 1, 320),       # K1: 16 splits (wide slab sum)
    (300, 20000, 5, 1, 20, 40, 512),       # K2: 40 splits (wide slab sum)
    (17000, 40, 3, 1, 1063, 1, 64),        # K1: one split over two flush segments
    (40, 17000, 3, 1, 3, 1, 17000),        # K2: one chunk over two flush segments
])
def test_componentwise_bound_against_exact_product(L, M, H, S1, kbs1, S2, kchunk):
    rng = np.random.default_rng(L + M)
    Y, B, A = _inputs(rng, L, M, H)
    plan = im.i8_round_plans(L, M, S1, kbs1, S2, kchunk)
    assert plan[0] * plan[1] >= L and plan[2] * plan[3] >= M
    P, Q = im.k1(Y, B, plan), im.k2(Y, A, plan)
    assert im.wide_sum(plan[0], M * H) == (plan[0] >= 16) and im.wide_sum(plan[2], H * ((L + 1) & ~1)) == (plan[2] >= 16)
    for i, h in zip(rng.integers(0, M, 25), rng.integers(0, H, 25)):
        ref = im.exact_dot(Y[:, i], B[:, h])
        assert abs(P[i, h] - ref) <= _bound_k1(Y, B, plan, i, h, ref), (i, h)
    for l, h in zip(rng.integers(0, L, 25), rng.integers(0, H, 25)):
        ref = im.exact_dot(Y[l, :], A[:, h])
        assert abs(Q[l, h] - ref) <= _bound_k2(Y, A, plan, l, h, ref), (l, h)
    # the bound stays far below what a wrong exponent (about W) or a lost low digit plane (about W 2^-55 per term) costs
    F, E = im.y_exponents(Y)
    G = im._masked_max(im.exp_digits(B) + F[:, None], B != 0, 0)
    assert _bound_k1(Y, B, plan, 0, 0, 0.0) < L * np.ldexp(1.0, int(E[0] + G[0])) * 2.0 ** -45


def test_model_sums_slabs_in_kernel_order():
    rng = np.random.default_rng(31)
    parts = [rng.standard_normal(50) * 10.0 ** rng.integers(-8, 9) for _ in range(21)]
    seq = 0.0 + parts[0]
    for p in parts[1:]:
        seq = seq + p
    assert np.array_equal(im.sum_partials(parts, 50 * 2 ** 15), seq)          # n > 2^20: sequential
    sub = [sum(parts[y::8][1:], 0.0 + parts[y]) for y in range(8)]
    wide = sub[0]
    for s in sub[1:]:
        wide = wide + s
    assert np.array_equal(im.sum_partials(parts, 50), wide)
    assert not np.array_equal(wide, seq)          # the two orders differ on this input, so the mode matters


def test_nonfinite_inputs_poison_exactly_their_rows_and_columns():
    rng = np.random.default_rng(32)
    Y, B, A = _inputs(rng, 40, 30, 5)
    Y[3, 7] = np.nan
    Y[11, 2] = np.inf
    B[5, 1] = -np.inf
    A[9, 4] = np.nan
    plan = (1, 64, 1, 32)
    P, Q = im.k1(Y, B, plan), im.k2(Y, A, plan)
    Pm = np.zeros(P.shape, bool)
    Pm[[7, 2], :] = True
    Pm[:, 1] = True
    Qm = np.zeros(Q.shape, bool)
    Qm[[3, 11], :] = True
    Qm[:, 4] = True
    assert np.array_equal(np.isnan(P), Pm) and np.array_equal(np.isnan(Q), Qm)
    Y0, B0, A0 = (np.where(np.isfinite(x), x, 0.0) for x in (Y, B, A))
    assert np.array_equal(P[~Pm], im.k1(Y0, B0, plan)[~Pm]) and np.array_equal(Q[~Qm], im.k2(Y0, A0, plan)[~Qm])


@pytest.mark.parametrize("seed", range(4))
def test_plan_rounding_covers_k_without_empty_splits(lib, seed):
    rng = np.random.default_rng(seed)
    for _ in range(200):
        L, M = int(rng.integers(1, 400000)), int(rng.integers(1, 400000))
        if rng.random() < 0.3:
            L, M = int(rng.integers(1, 300)), int(rng.integers(1, 300))
        H = int(rng.integers(1, 65))
        sms = int(rng.choice([148, 132, 1, 7]))
        S1, klen, S2, kchunk = im.i8_plans(lib, L, M, H, sms)
        assert klen % 32 == 0 and kchunk % 32 == 0
        assert S1 * klen >= L and (S1 - 1) * klen < L, (L, M, H, sms)
        assert S2 * kchunk >= M and (S2 - 1) * kchunk < M, (L, M, H, sms)
