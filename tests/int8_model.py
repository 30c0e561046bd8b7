"""Bit-exact NumPy model of the INT8 contractions (csrc/gemm_int8.cu) as `gemm_YtB` / `gemm_YA` run them.

Where tools/int8gemm/emulate_ozaki.py models the scheme's error level, this module repeats the kernel's arithmetic operation
for operation, so its output is compared with the GPU's by `np.array_equal`:
  exponents   F_l: frexp exponent of the row maximum; E_m: smallest e with |Y_lm 2^-F_l| <= (127/128) 2^e over the column;
              K1 operand G_h = max_l e(B_lh) + F_l, K2 operand G_ch = max_{m in chunk c} e(A_mh) + E_m (127/128 rule);
              an all-zero line gets 0.  Exponents are combined as integers, never by rescaling the data.
  digits      X = rint(ldexp(x, 55 - e)) (ties to even), seven balanced radix-256 digits taken from the bottom.
  split plan  vbmf_b200_plan_contractions, rounded as i8_plans (csrc/capi.cu) rounds it.
  levels      per work item (tile, split) and per 16384-k flush segment: level k = sum_{i+j=k} digit-plane products, exact
              in float64 BLAS (|level| < 2^31).
  combination acc = acc * 2^-8 + level_k from level 6 down to 0, then ldexp(acc, rowexp + colexp - 14); flush segments are
              added in order into the slab.
  slab sum    sum_partials (csrc/kernels.cu): sequential from 0.0, or 8 strided subsets combined in order when S >= 16
              and n <= 2^20.
Non-finite inputs: the model runs on the inputs with NaN / Inf replaced by 0, then writes NaN into every output row and
column that a non-finite input reaches, as the kernel's epilogue does.
"""
import numpy as np

NSL = 7
DIGIT_MAX = 127.0 / 128.0
SEG_K = 16384          # k per INT32 flush segment


# ------------------------------------------------------------------------------------------- exponents and digits
def exp_frexp(x):
    """frexp exponent per element (callers mask zeros themselves)."""
    return np.frexp(x)[1].astype(np.int64)


def exp_digits(x):
    """smallest e with |x| <= (127/128) 2^e (frexp's exponent, plus one when the mantissa exceeds 127/128)."""
    m, e = np.frexp(x)
    return (e + (np.abs(m) > DIGIT_MAX)).astype(np.int64)


def _masked_max(e, nz, axis):
    """max of e over the nonzero entries along axis; 0 where a line is all zero (exp_fix)."""
    lo = np.iinfo(np.int64).min
    r = np.max(np.where(nz, e, lo), axis=axis)
    return np.where(r == lo, 0, r)


def y_exponents(Y):
    """F[L] (frexp rule on the row maxima) and E[M] (127/128 rule on the row-scaled columns)."""
    nz = Y != 0
    F = _masked_max(exp_frexp(Y), nz, 1)
    E = _masked_max(exp_digits(Y) - F[:, None], nz, 0)
    return F, E


def fixed55(x, e):
    """rint(x * 2^(55 - e)) as int64, one rounding (ties to even)."""
    return np.rint(np.ldexp(x, 55 - e)).astype(np.int64)


def digits(X):
    """balanced radix-256 digits of the int64 array X, most significant first (digit i weighs 2^-(7+8i) of X/2^55)."""
    X = np.asarray(X, np.int64).copy()
    D = []
    for _ in range(NSL):
        d = ((X + 128) & 255) - 128
        X = (X - d) >> 8
        D.append(d)
    assert not np.any(X), "value outside the range of seven balanced digits"
    return [d.astype(np.int8) for d in D[::-1]]


# ------------------------------------------------------------------------------------------- plan
def i8_plans(lib, L, M, H, num_sms):
    """(S1, klen1, S2, kchunk): the FP64 plan of vbmf_b200_plan_contractions rounded as i8_plans in csrc/capi.cu."""
    out = np.zeros(6, np.int64)
    rc = lib.vbmf_b200_plan_contractions(L, M, H, num_sms, out.ctypes.data)
    assert rc == 0
    S1, kbs1, S2, kchunk = (int(v) for v in out[:4])
    return i8_round_plans(L, M, S1, kbs1, S2, kchunk)


def i8_round_plans(L, M, S1, kbs1, S2, kchunk):
    kbs1 = (kbs1 + 1) & ~1
    nkb = (L + 15) // 16
    S1 = max(1, -(-nkb // kbs1))
    kchunk = -(-kchunk // 32) * 32
    S2 = max(1, -(-M // kchunk))
    return S1, kbs1 * 16, S2, kchunk


# ------------------------------------------------------------------------------------------- the contraction
def _levels_combined(DA, DB, k0, k1, rowexp, colexp):
    """one flush segment [k0, k1): levels 0..6 of the digit planes DA [k][rows], DB [k][H], combined and scaled."""
    lev = [np.zeros((DA[0].shape[1], DB[0].shape[1])) for _ in range(NSL)]
    b = [d[k0:k1].astype(np.float64) for d in DB]
    for i in range(NSL):
        a = DA[i][k0:k1].astype(np.float64)
        for j in range(NSL - i):
            lev[i + j] += a.T @ b[j]                  # integers below 2^31: float64 BLAS is exact
    acc = lev[NSL - 1]
    for k in range(NSL - 2, -1, -1):
        acc = acc * 2.0 ** -8 + lev[k]                 # the kernel's fma(acc, 2^-8, level_k): one rounding
    return np.ldexp(acc, rowexp[:, None] + colexp[None, :] - 14)


def _slab(DA, DB, k0, k1, rowexp, colexp):
    out = None
    for g0 in range(k0, k1, SEG_K):
        x = _levels_combined(DA, DB, g0, min(k1, g0 + SEG_K), rowexp, colexp)
        out = x if out is None else out + x
    return out


def sum_partials(parts, n):
    """csrc/kernels.cu sum_partials on S equal-shape partials; n is the element count the caller passes (it picks the mode)."""
    S = len(parts)
    if wide_sum(S, n):
        sub = []
        for y in range(8):
            s = np.zeros_like(parts[0])
            for p in range(y, S, 8):
                s = s + parts[p]
            sub.append(s)
        t = sub[0]
        for k in range(1, 8):
            t = t + sub[k]
        return t
    s = np.zeros_like(parts[0])
    for p in parts:
        s = s + p
    return s


def wide_sum(S, n):
    """True when sum_partials takes the 8-subset mode."""
    return S >= 16 and n <= 1 << 20


def _clean(x):
    x = np.array(x, dtype=np.float64, order="F")
    bad = ~np.isfinite(x)
    x[bad] = 0.0
    return x, bad


def row_exponents(Y, block=4096):
    """F[L] of a finite Y, in column blocks (for matrices too large for whole-array temporaries)."""
    mx = np.zeros(Y.shape[0])
    for m0 in range(0, Y.shape[1], block):
        mx = np.maximum(mx, np.max(np.abs(Y[:, m0:m0 + block]), axis=1))
    return np.where(mx == 0, 0, exp_frexp(mx))


def k1(Y, B, plan, cols=None):
    """P = Y' B (M x H) as gemm_YtB computes it on the INT8 path; plan = i8_plans(...).  With cols (an index array of Y's
    columns), only those rows of P, in that order: F still comes from the whole Y."""
    n_sum = max(Y.shape[1], 1) * B.shape[1]          # the element count sum_partials is called with
    if cols is not None:
        F = row_exponents(Y)
        Y = Y[:, cols]
    Y, ybad = _clean(Y)
    B, bbad = _clean(B)
    L, M = Y.shape
    H = B.shape[1]
    S1, klen = plan[0], plan[1]
    if cols is None:
        F, E = y_exponents(Y)
    else:
        E = _masked_max(exp_digits(Y) - F[:, None], Y != 0, 0)
    G = _masked_max(exp_digits(B) + F[:, None], B != 0, 0)
    DY = digits(fixed55(Y, F[:, None] + E[None, :]))
    DB = digits(fixed55(B, G[None, :] - F[:, None]))
    slabs = [_slab(DY, DB, s * klen, min(L, (s + 1) * klen), E, G) for s in range(S1)]
    P = slabs[0] if S1 == 1 else sum_partials(slabs, n_sum)
    P[np.any(ybad, axis=0), :] = np.nan
    P[:, np.any(bbad, axis=0)] = np.nan
    return P


def k2(Y, A, plan):
    """Q = Y A (L x H) as gemm_YA computes it on the INT8 path; plan = i8_plans(...)."""
    Y, ybad = _clean(Y)
    A, abad = _clean(A)
    L, M = Y.shape
    H = A.shape[1]
    S, kchunk = plan[2], plan[3]
    F, E = y_exponents(Y)
    DY = digits(fixed55(Y.T, E[:, None] + F[None, :]))     # [m][l]: k = m
    slabs = []
    for c in range(S):
        m0, m1 = c * kchunk, min(M, (c + 1) * kchunk)
        Ac = A[m0:m1]
        Gc = _masked_max(exp_digits(Ac) + E[m0:m1, None], Ac != 0, 0)
        DA = digits(fixed55(Ac, Gc[None, :] - E[m0:m1, None]))
        slabs.append(_slab([d[m0:m1] for d in DY], DA, 0, m1 - m0, F, Gc))     # flush segments start at the chunk
    Q = sum_partials(slabs, H * ((L + 1) & ~1))
    Q[np.any(ybad, axis=1), :] = np.nan
    Q[:, np.any(abad, axis=0)] = np.nan
    return Q


# ------------------------------------------------------------------------------------------- exact reference
def _two_prod(a, b):
    """Dekker: a * b = p + e exactly (no overflow or underflow in the split)."""
    p = a * b
    c = 134217729.0
    ah = a * c
    ah = ah - (ah - a)
    al = a - ah
    bh = b * c
    bh = bh - (bh - b)
    bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_dot(x, y):
    """the exactly rounded sum_i x_i y_i (math.fsum of the exact two-products)."""
    import math
    p, e = _two_prod(np.asarray(x, np.float64), np.asarray(y, np.float64))
    return math.fsum(np.concatenate([p, e]).tolist())
