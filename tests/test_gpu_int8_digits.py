"""K1 / K2 on the INT8 path (csrc/gemm_int8.cu) at the edges of the signed radix-256 digits: level 6 near its INT32 bound
across the 16384-k flush, and column maxima on both sides of 127/128, where the exponent rule adds one."""
import os
import sys

import numpy as np
import pytest

from tests.test_gpu_int8_gemm import _exact_err

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "int8gemm"))
import emulate_ozaki as oz  # noqa: E402

pytestmark = pytest.mark.gpu

EDGE = 127.0 / 128.0


@pytest.fixture(scope="module")
def G():
    from tests import gpu_helpers
    return gpu_helpers


@pytest.fixture(scope="module")
def ctx(G):
    c = G.vb.Context(device=0)
    yield c
    c.close()


def _value(digits):
    """the float64 whose digits in the model are exactly `digits` (most significant first)"""
    w = float(sum(int(d) * 256 ** (6 - i) for i, d in enumerate(digits))) * 2.0 ** -55
    F, E, Z = oz.scale_Y_digits(np.array([[w]]))
    assert F[0] == 0 and E[0] == 0 and [int(d[0, 0]) for d in oz.split_digits(Z)] == list(digits)
    return w


# |Z| <= 127/128 keeps the top digit off -128: these digits put level 6 at 2*126*124 + 5*127^2 = 111893 per k, 97.6 % of
# 7 * 128^2, so without the flush every 16384 k it wraps past 2^31 after 19193 k
W_MAX = _value([126, 127, 127, 127, 127, 127, 124])


def _signs(rng, n):
    return np.where(rng.random(n) < 0.5, -1.0, 1.0)


# At these shapes a 148-SM B200 runs the contraction under test as a single split: one 128-row tile per SM, the whole
# k = 20480 in one work item, so the INT32 accumulators must be flushed once.
@pytest.mark.parametrize("which", ["k1", "k2"])
def test_int8_level6_bound_across_flush(G, ctx, which):
    rows, k, H = 18944, 20480, 64
    rng = np.random.default_rng(31 if which == "k1" else 32)
    s, t, u = _signs(rng, k), _signs(rng, rows), _signs(rng, H)
    # rank-one sign patterns: every product of a contraction sum has the same sign, so every level sum grows with k
    if which == "k1":
        Y = np.outer(t * W_MAX, s).T          # L = k, M = rows, Fortran order
        B = np.asfortranarray(np.outer(s, u) * W_MAX)
        ctx.attach(Y, force=True)
        P, Pr = ctx.gemm_YtB(B), Y.T @ B
        assert G.rel(P, Pr) < 1e-13
        assert _exact_err(P, Y.T, B) <= 4 * max(_exact_err(Pr, Y.T, B), 1e-16 * np.max(np.abs(Pr)))
    else:
        Y = np.outer(s * W_MAX, t).T          # L = rows, M = k, Fortran order
        A = np.outer(s, u) * W_MAX
        ctx.attach(Y, force=True)
        Q, Qr = ctx.gemm_YA(A), Y @ A
        assert G.rel(Q, Qr) < 1e-13
        assert _exact_err(Q, Y, A) <= 4 * max(_exact_err(Qr, Y, A), 1e-16 * np.max(np.abs(Qr)))


def _bumped(rng, n, k):
    """n x k values in (-0.9, 0.9) whose column maxima sit just above 127/128, just below it, exactly on it, or at 1 - 2^-53,
    with random signs"""
    X = rng.uniform(-0.9, 0.9, (n, k))
    edge = np.array([np.nextafter(EDGE, 1), np.nextafter(EDGE, 0), EDGE, 1 - 2.0 ** -53])
    X[rng.integers(0, n, k), np.arange(k)] = edge[np.arange(k) % 4] * _signs(rng, k)
    return X


@pytest.mark.parametrize("L,M,H", [(1000, 3001, 33), (4099, 20000, 64)])
def test_int8_exponent_bump(G, ctx, L, M, H):
    rng = np.random.default_rng(L + M + H)
    # Y: column maxima at the edges after row scaling; powers of two per row and column move every exponent, not the bump
    r, c = rng.integers(-20, 21, L), rng.integers(-20, 21, M)
    Y = np.asfortranarray(np.ldexp(_bumped(rng, L, M), r[:, None] + c[None, :]))
    # operands: diag(2^F) B has the edge column maxima; diag(2^E) A has them up to the factor 2 of Y's own bump
    B = np.asfortranarray(np.ldexp(_bumped(rng, L, H), -r[:, None]))
    A = np.ldexp(_bumped(rng, M, H), -c[:, None])
    ctx.attach(Y, force=True)
    P, Q = ctx.gemm_YtB(B), ctx.gemm_YA(A)
    assert G.rel(P, Y.T @ B) < 1e-13 and G.rel(Q, Y @ A) < 1e-13
