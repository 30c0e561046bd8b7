"""NumPy models of the INT8 contractions (csrc/gemm_int8.cu): two-sided power-of-two scaling, the operands cut into int8
digit planes, level sums i + j = k in exact integers, levels combined in float64 from the last down to 0.

Two schemes:
  8 x 7-bit   eight truncated 7-bit slices in [-127, 127], levels 0..7 (36 slice products): the earlier kernel, kept here as
              the comparator (split, k1, k2).
  7 x 8-bit   seven balanced radix-256 digits in [-128, 127] of rint(Z * 2^55), |Z| <= 127/128, levels 0..6 (28 slice
              products): what the kernel runs (split_digits, k1_digits, k2_digits).

    python tools/int8gemm/emulate_ozaki.py     # normwise error of the schemes against an all-pairs 10-slice product

The 7-bit table is what fixed the earlier scheme at 8 slices: 7 slices leave a normwise error around 1e-13, 8 come within a
small factor of the float64 product's own error.  Seven 8-bit digits carry the same 56 bits with 28 products instead of 36.
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


def slice_matmul(S, T):
    """S' T of int8-range slices, exact: every partial sum is an integer below 2^14 k < 2^53, so float64 BLAS is exact."""
    assert S.shape[0] < 2 ** 39
    return (S.T.astype(np.float64) @ T.astype(np.float64)).astype(np.int64)


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
                levels[i + j] += slice_matmul(SY[i], SB[j])
    return np.ldexp(combine(levels), E[:, None] + G[None, :])


def k2(Y, A, **kw):
    """Q = Y A: the same scheme with the roles of rows and columns exchanged."""
    return k1(np.ascontiguousarray(Y.T), A, **kw)


# ------------------------------------------------------------------------------------------- 7 x 8-bit signed digits
DIGITS = 7
DIGIT_MAX = 127.0 / 128.0   # |Z| bound that keeps rint(Z * 2^55) inside the range of seven balanced digits


def exponent_digits(x):
    """smallest e with |x| <= (127/128) 2^e per element (frexp's exponent, plus one above 127/128); 0 for zeros."""
    m, e = np.frexp(x)
    e = e + (np.abs(m) > DIGIT_MAX)
    return np.where(x == 0, 0, e).astype(np.int64)


def max_exponent_digits(x, axis):
    """exponent_digits of the maximum along axis (the rule is monotonic in |x|); 0 for an all-zero line."""
    return exponent_digits(np.max(np.abs(x), axis=axis))


def scale_Y_digits(Y):
    """F (rows, frexp rule), E (columns, 127/128 rule) with Z = 2^-F Y 2^-E, |Z| <= 127/128."""
    F = max_exponent(Y, 1)
    Yr = np.ldexp(Y, -F[:, None])
    E = max_exponent_digits(Yr, 0)
    return F, E, np.ldexp(Yr, -E[None, :])


def digits_of(X, n=DIGITS):
    """balanced radix-256 digits of the integers X, taken from the bottom: d = ((X + 128) & 255) - 128, X = (X - d) >> 8.
    Returns the digits most significant first (X = sum_i d_i 256^(n-1-i) + 256^n rest) and what is left of X."""
    X = np.asarray(X, np.int64).copy()
    D = []
    for _ in range(n):
        d = ((X + 128) & 255) - 128
        X = (X - d) >> 8
        D.append(d)
    return D[::-1], X


def split_digits(Z, n=DIGITS):
    """Z = sum_i 2^-(7+8i) D_i + r, D_i in [-128, 127], |r| <= 2^-56 (|Z| <= 127/128)."""
    D, rest = digits_of(np.rint(np.ldexp(Z, 55)).astype(np.int64), n)
    assert not np.any(rest), "value outside the range of the digits"
    return D


def combine_digits(levels):
    """sum_k 2^-(8k+14) level_k, levels 6 down to 0 (the kernel's order)."""
    acc = levels[-1].astype(np.float64)
    for k in range(len(levels) - 2, -1, -1):
        acc = acc * 2.0 ** -8 + levels[k].astype(np.float64)
    return acc * 2.0 ** -14


def k1_digits(Y, B, cut=DIGITS - 1):
    """P = Y' B through the signed-digit scheme (levels 0..cut)."""
    F, E, Z = scale_Y_digits(Y)
    Bs = np.ldexp(B, F[:, None])
    G = max_exponent_digits(Bs, 0)
    W = np.ldexp(Bs, -G[None, :])
    DY, DB = split_digits(Z), split_digits(W)
    levels = [np.zeros((Y.shape[1], B.shape[1]), np.int64) for _ in range(cut + 1)]
    for i in range(DIGITS):
        for j in range(DIGITS):
            if i + j <= cut:
                levels[i + j] += slice_matmul(DY[i], DB[j])
    return np.ldexp(combine_digits(levels), E[:, None] + G[None, :])


def k2_digits(Y, A, **kw):
    """Q = Y A through the signed-digit scheme."""
    return k1_digits(np.ascontiguousarray(Y.T), A, **kw)


def rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def main_cases():
    """the three (Y, B, A) inputs main() reports on"""
    rng = np.random.default_rng(7)
    for L, M, rowscale in ((2000, 1000, False), (1500, 1500, False), (1500, 1500, True)):
        U = rng.standard_normal((L, 32))
        V = rng.standard_normal((32, M))
        Y = U @ V / np.sqrt(32) + 0.1 * rng.standard_normal((L, M))
        if rowscale:
            Y = np.ldexp(Y, rng.integers(-12, 13, L)[:, None])
        B = rng.standard_normal((L, 64)) * np.exp(rng.uniform(-6, 2, 64))[None, :]
        A = rng.standard_normal((M, 64)) * np.exp(rng.uniform(-6, 2, 64))[None, :]
        yield L, M, rowscale, Y, B, A


def main():
    for L, M, rowscale, Y, B, A in main_cases():
        refP = k1(Y, B, ns_y=10, ns_b=10, cut=18)
        refQ = k2(Y, A, ns_y=10, ns_b=10, cut=18)
        row = {"shape": (L, M), "row_scales": rowscale,
               "fp64": (rel(Y.T @ B, refP), rel(Y @ A, refQ)),
               "7+7": (rel(k1(Y, B, ns_y=7, ns_b=7, cut=6), refP), rel(k2(Y, A, ns_y=7, ns_b=7, cut=6), refQ)),
               "8+8": (rel(k1(Y, B), refP), rel(k2(Y, A), refQ)),
               "7x8bit": (rel(k1_digits(Y, B), refP), rel(k2_digits(Y, A), refQ))}
        print({k: (tuple("%.1e" % x for x in v) if isinstance(v, tuple) and isinstance(v[0], float) else v) for k, v in row.items()})


if __name__ == "__main__":
    main()
