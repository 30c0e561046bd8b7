"""K1 / K2 on the INT8 slice path (csrc/gemm_int8.cu, H <= 64) against NumPy, an exact integer reference and the FP64
tensor-core path (VBMF_B200_GEMM=dmma)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    from tests import gpu_helpers
    return gpu_helpers


@pytest.fixture(scope="module")
def ctx(G):
    c = G.vb.Context(device=0)
    yield c
    c.close()


def _scaled(rng, L, M):
    Y = rng.standard_normal((L, M))
    Y *= np.ldexp(1.0, rng.integers(-30, 31, L))[:, None] * np.ldexp(1.0, rng.integers(-30, 31, M))[None, :]
    Y[L // 2, :] = 0.0
    Y[:, M // 3] = 0.0
    return np.asfortranarray(Y)


def _exact_err(X, Z, Wt):
    """normwise error of X against the exactly rounded product Z @ Wt (integer arithmetic on the float64 mantissas)."""
    from fractions import Fraction
    rng = np.random.default_rng(0)
    idx = [(int(i), int(j)) for i, j in zip(rng.integers(0, X.shape[0], 20), rng.integers(0, X.shape[1], 20))]
    worst = 0.0
    for i, j in idx:
        ref = float(sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(Z[i, :], Wt[:, j])))
        worst = max(worst, abs(X[i, j] - ref))
    return worst


@pytest.mark.parametrize("L,M,H", [(1000, 3001, 1), (257, 1000, 7), (513, 777, 33), (3000, 50000, 64), (40000, 300, 64)])
def test_int8_contractions_scaled(G, ctx, L, M, H):
    rng = np.random.default_rng(L + 3 * M + H)
    Y = _scaled(rng, L, M)
    B = np.asfortranarray(rng.standard_normal((L, H)) * np.exp(rng.uniform(-6, 2, H))[None, :])
    A = np.asfortranarray(rng.standard_normal((M, H)) * np.exp(rng.uniform(-6, 2, H))[None, :])
    ctx.attach(Y, force=True)
    P, Q = ctx.gemm_YtB(B), ctx.gemm_YA(A)
    Pr, Qr = Y.T @ B, Y @ A
    assert G.rel(P, Pr) < 1e-13 and G.rel(Q, Qr) < 1e-13
    # against the exact product: at most 4x the float64 product's own error (sampled entries, normwise)
    assert _exact_err(P, Y.T, B) <= 4 * max(_exact_err(Pr, Y.T, B), 1e-16 * np.max(np.abs(Pr)))
    assert _exact_err(Q, Y, A) <= 4 * max(_exact_err(Qr, Y, A), 1e-16 * np.max(np.abs(Qr)))
    assert np.array_equal(P, ctx.gemm_YtB(B)) and np.array_equal(Q, ctx.gemm_YA(A))


def test_int8_flush_beyond_16384(G, ctx):
    # every slice of Y and of the operands at +-127: level 7 reaches its bound, so K1 (k = L = 40000) and K2 (k = M) must flush
    L, M, H = 40000, 20000, 16
    rng = np.random.default_rng(5)
    v = 1.0 - 2.0 ** -52
    Y = np.asfortranarray(np.where(rng.random((L, M)) < 0.5, -v, v))
    Y[:, 0] = v
    B = np.asfortranarray(np.full((L, H), v))
    A = np.full((M, H), v)
    ctx.attach(Y, force=True)
    P, Q = ctx.gemm_YtB(B), ctx.gemm_YA(A)
    assert G.rel(P, Y.T @ B) < 1e-13 and G.rel(Q, Y @ A) < 1e-13


@pytest.mark.parametrize("L,M,H", [(50000, 1000, 64), (999, 70001, 33), (17, 5, 7)])
def test_int8_integer_inputs_exact(G, ctx, L, M, H):
    rng = np.random.default_rng(L * M)
    Y = np.asfortranarray(rng.integers(-1000, 1001, (L, M)).astype(np.float64))
    B = np.asfortranarray(rng.integers(-100, 101, (L, H)).astype(np.float64))
    A = np.asfortranarray(rng.integers(-100, 101, (M, H)).astype(np.float64))
    ctx.attach(Y, force=True)
    assert np.array_equal(ctx.gemm_YtB(B), Y.T @ B)
    assert np.array_equal(ctx.gemm_YA(A), Y @ A)


def test_int8_agrees_with_dmma(G):
    rng = np.random.default_rng(11)
    L, M, H = 2048, 20000, 64
    Y = np.asfortranarray(rng.standard_normal((L, M)))
    B = np.asfortranarray(rng.standard_normal((L, H)))
    A = np.asfortranarray(rng.standard_normal((M, H)))
    out = {}
    old = os.environ.get("VBMF_B200_GEMM")
    try:
        for path in ("int8", "dmma"):
            if path == "dmma":
                os.environ["VBMF_B200_GEMM"] = "dmma"
            else:
                os.environ.pop("VBMF_B200_GEMM", None)
            c = G.vb.Context(device=0)
            c.attach(Y, force=True)
            out[path] = (c.gemm_YtB(B), c.gemm_YA(A))
            c.close()
    finally:
        if old is None:
            os.environ.pop("VBMF_B200_GEMM", None)
        else:
            os.environ["VBMF_B200_GEMM"] = old
    assert G.rel(out["int8"][0], out["dmma"][0]) < 1e-13
    assert G.rel(out["int8"][1], out["dmma"][1]) < 1e-13
