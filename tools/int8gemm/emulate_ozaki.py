"""NumPy model of the INT8 contractions (csrc/gemm_int8.cu): two-sided power-of-two scaling, eight truncated 7-bit slices
per operand, level sums i + j = k in exact integers, levels 7 down to 0 combined in float64.

    python tools/int8gemm/emulate_ozaki.py     # normwise error of the slice schemes against an all-pairs 10-slice product

The printed table is what fixed the scheme at 8 slices per operand and levels 0..7 (36 slice products): 7 slices leave a
normwise error around 1e-13, 8 slices come within a small factor of the float64 product's own error.
"""
import numpy as np

NSL = 8


def exponent(x):
    """frexp exponent per element (|x| < 2^e); 0 for zeros."""
    _, e = np.frexp(x)
    return np.where(x == 0, 0, e).astype(np.int64)


def max_exponent(x, axis):
    """exponent of the maximum along axis; 0 for an all-zero line."""
    return exponent(np.max(np.abs(x), axis=axis))


def scale_Y(Y):
    """F (rows), E (columns) with Z = 2^-F Y 2^-E, |Z| < 1."""
    F = max_exponent(Y, 1)
    Yr = np.ldexp(Y, -F[:, None])
    E = max_exponent(Yr, 0)
    return F, E, np.ldexp(Yr, -E[None, :])


def split(Z, nsl=NSL):
    """truncated 7-bit slices: Z = sum_i 128^-(i+1) S_i + r, |S_i| <= 127, |r| < 128^-nsl (|Z| < 1)."""
    t = Z.copy()
    S = []
    for _ in range(nsl):
        t = t * 128.0
        s = np.trunc(t)
        t = t - s
        S.append(s.astype(np.int64))
    return S


def combine(levels):
    """sum_k 2^-7(k+2) level_k, levels 7 down to 0 (the kernel's order)."""
    acc = levels[-1].astype(np.float64)
    for k in range(len(levels) - 2, -1, -1):
        acc = acc * 2.0 ** -7 + levels[k].astype(np.float64)
    return acc * 2.0 ** -14


def k1(Y, B, ns_y=NSL, ns_b=NSL, cut=NSL - 1):
    """P = Y' B through the slice scheme (levels 0..cut)."""
    F, E, Z = scale_Y(Y)
    Bs = np.ldexp(B, F[:, None])
    G = max_exponent(Bs, 0)
    W = np.ldexp(Bs, -G[None, :])
    SY, SB = split(Z, ns_y), split(W, ns_b)
    levels = [np.zeros((Y.shape[1], B.shape[1]), np.int64) for _ in range(cut + 1)]
    for i in range(ns_y):
        for j in range(ns_b):
            if i + j <= cut:
                levels[i + j] += SY[i].T @ SB[j]
    return np.ldexp(combine(levels), E[:, None] + G[None, :])


def k2(Y, A, **kw):
    """Q = Y A: the same scheme with the roles of rows and columns exchanged."""
    return k1(np.ascontiguousarray(Y.T), A, **kw)


def rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def main():
    rng = np.random.default_rng(7)
    for L, M, rowscale in ((2000, 1000, False), (1500, 1500, False), (1500, 1500, True)):
        U = rng.standard_normal((L, 32))
        V = rng.standard_normal((32, M))
        Y = U @ V / np.sqrt(32) + 0.1 * rng.standard_normal((L, M))
        if rowscale:
            Y = np.ldexp(Y, rng.integers(-12, 13, L)[:, None])
        B = rng.standard_normal((L, 64)) * np.exp(rng.uniform(-6, 2, 64))[None, :]
        A = rng.standard_normal((M, 64)) * np.exp(rng.uniform(-6, 2, 64))[None, :]
        refP = k1(Y, B, ns_y=10, ns_b=10, cut=18)
        refQ = k2(Y, A, ns_y=10, ns_b=10, cut=18)
        row = {"shape": (L, M), "row_scales": rowscale,
               "fp64": (rel(Y.T @ B, refP), rel(Y @ A, refQ)),
               "7+7": (rel(k1(Y, B, ns_y=7, ns_b=7, cut=6), refP), rel(k2(Y, A, ns_y=7, ns_b=7, cut=6), refQ)),
               "8+8": (rel(k1(Y, B), refP), rel(k2(Y, A), refQ))}
        print({k: (tuple("%.1e" % x for x in v) if isinstance(v, tuple) and isinstance(v[0], float) else v) for k, v in row.items()})


if __name__ == "__main__":
    main()
