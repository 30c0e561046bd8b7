"""K1 / K2 on the INT8 path bit for bit against the host model of tests/int8_model.py, the non-finite rule of that path, and
the spectral norm of the convergence test at the ends of the double range.

Every contraction case compares `ctx.gemm_YtB` / `ctx.gemm_YA` with the model by `np.array_equal` (NaN equal to NaN): an
error confined to small entries, one split-K chunk, one flush segment or one work item of a persistent CTA shows up here,
where the normwise checks of test_gpu_int8_gemm.py would let it pass."""
import os
import warnings

import numpy as np
import pytest

from tests import int8_model as im

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


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _plan(G, L, M, H, num_sms):
    return im.i8_plans(G.vb._lib.load(), L, M, H, num_sms)


def _same(x, ref):
    return x.shape == ref.shape and np.array_equal(x, ref, equal_nan=True)


def _check(G, ctx, num_sms, Y, B, A, attach=True):
    """attach Y (unless already resident), run both contractions, compare with the model; returns the plan"""
    if attach:
        ctx.attach(Y)
    L, M = Y.shape
    plan = _plan(G, L, M, B.shape[1], num_sms)
    P, Q = ctx.gemm_YtB(B), ctx.gemm_YA(A)
    Pm, Qm = im.k1(Y, B, plan), im.k2(Y, A, plan)
    assert _same(P, Pm), "K1 differs from the model at %d entries (L=%d M=%d H=%d)" % (np.sum(~((P == Pm) | (np.isnan(P) & np.isnan(Pm)))), L, M, B.shape[1])
    assert _same(Q, Qm), "K2 differs from the model at %d entries (L=%d M=%d H=%d)" % (np.sum(~((Q == Qm) | (np.isnan(Q) & np.isnan(Qm)))), L, M, A.shape[1])
    return plan


def _inputs(rng, L, M, H):
    Y = rng.standard_normal((L, M)) * np.ldexp(1.0, rng.integers(-30, 31, L))[:, None] * np.ldexp(1.0, rng.integers(-30, 31, M))[None, :]
    if L > 2 and M > 2:            # an all-zero row and column next to data (at L or M <= 2 they would be most or all of Y)
        Y[L // 2, :] = 0.0
        Y[:, M // 3] = 0.0
    B = rng.standard_normal((L, H)) * np.ldexp(1.0, rng.integers(-20, 21, H))[None, :]
    A = rng.standard_normal((M, H)) * np.ldexp(1.0, rng.integers(-20, 21, H))[None, :]
    return np.asfortranarray(Y), np.asfortranarray(B), np.asfortranarray(A)


# ------------------------------------------------------------------------------------------- shapes
def test_every_H_from_1_to_64(G, ctx, num_sms):
    # Hp = 16 / 32 / 48 / 64: tensor-memory allocations of 128 / 256 / 512 columns, N pieces cut at 256 (Hp = 48: 256 + 80)
    rng = np.random.default_rng(1)
    L, M = 129, 161
    Y, B, A = _inputs(rng, L, M, 64)
    ctx.attach(Y)
    for H in range(1, 65):
        _check(G, ctx, num_sms, Y, np.asfortranarray(B[:, :H]), np.asfortranarray(A[:, :H]), attach=False)


@pytest.mark.parametrize("H", [7, 64])
def test_small_and_ragged_shapes(G, ctx, num_sms, H):
    sizes = (1, 2, 15, 16, 17, 31, 32, 33, 127, 128, 129)
    rng = np.random.default_rng(H)
    for L in sizes:
        for M in sizes:
            Y, B, A = _inputs(rng, L, M, H)
            assert np.any(Y) and np.any(B) and np.any(A)
            if L <= 2 or M <= 2:                                # no zero line: every row and column carries data
                assert np.all(Y != 0)
            _check(G, ctx, num_sms, Y, B, A)


# ------------------------------------------------------------------------------------------- pipeline structure
def test_k2_several_items_per_cta_wide_sum_and_chunk_exponents(G, ctx, num_sms):
    L, M, H = 1200, 20000, 16
    rng = np.random.default_rng(2)
    Y, B, A = _inputs(rng, L, M, H)
    S1, klen, S, kchunk = _plan(G, L, M, H, num_sms)
    # A's split-K chunks alternate between scales 2^0 and 2^45: the operand exponents of one column differ by >= 2^40
    A *= np.ldexp(1.0, 45 * ((np.arange(M) // kchunk) % 2))[:, None]
    ntile = (L + 127) // 128
    assert ntile * S > num_sms and M % kchunk != 0            # some CTA walks two work items; the last split is ragged
    assert S >= 16 and im.wide_sum(S, H * ((L + 1) & ~1))      # the 8-subset slab sum runs
    F, E = im.y_exponents(Y)
    Gc = [im._masked_max(im.exp_digits(A[c * kchunk:(c + 1) * kchunk]) + E[c * kchunk:(c + 1) * kchunk, None],
                         A[c * kchunk:(c + 1) * kchunk] != 0, 0) for c in range(S)]
    assert np.all(np.max(Gc, axis=0) - np.min(Gc, axis=0) >= 40)
    assert (M + 127) // 128 * S1 > num_sms                      # K1 too walks several items per CTA
    _check(G, ctx, num_sms, Y, B, A)


def test_k1_several_items_per_cta_and_wide_sum(G, ctx, num_sms):
    L, M, H = 40000, 1200, 8
    Y, B, A = _inputs(np.random.default_rng(3), L, M, H)
    S1, klen, S, kchunk = _plan(G, L, M, H, num_sms)
    assert (M + 127) // 128 * S1 > num_sms and L % klen != 0
    assert S1 >= 16 and im.wide_sum(S1, M * H)
    _check(G, ctx, num_sms, Y, B, A)


def test_k1_flush_segments_inside_persistent_ctas(G, ctx, num_sms):
    # klen > 16384: every work item spans two flush segments, while the grid walks 160 items on num_sms CTAs.  The model
    # runs on tile 0 and tile 8 (CTA 0's first and second item at 148 SMs) and the ragged last tile only.
    L, M, H = 263000, 1160, 3
    rng = np.random.default_rng(4)
    Y = rng.standard_normal((M, L)).T                          # Fortran order without a copy
    Y *= np.ldexp(1.0, rng.integers(-20, 21, M))[None, :]
    B = np.asfortranarray(rng.standard_normal((L, H)))
    S1, klen, S, kchunk = _plan(G, L, M, H, num_sms)
    ntile = (M + 127) // 128
    assert klen > im.SEG_K and ntile * S1 > num_sms
    w2 = num_sms                                                # CTA 0's second work item
    tiles = sorted({0, w2 % ntile, ntile - 1})
    cols = np.concatenate([np.arange(t * 128, min(M, t * 128 + 128)) for t in tiles])
    ctx.attach(Y)
    P = ctx.gemm_YtB(B)
    assert _same(P[cols], im.k1(Y, B, (S1, klen, S, kchunk), cols=cols))
    ctx.attach(np.zeros((1, 1)))                               # release the large Y


# ------------------------------------------------------------------------------------------- magnitudes
@pytest.mark.parametrize("L,M", [(129, 161), (2000, 3001)])
def test_scales_up_to_2_pow_1000(G, ctx, num_sms, L, M):
    rng = np.random.default_rng(L)
    H = 7
    r, c = rng.integers(-500, 501, L), rng.integers(-500, 501, M)
    Y = np.asfortranarray(rng.standard_normal((L, M)) * np.ldexp(1.0, r)[:, None] * np.ldexp(1.0, c)[None, :])
    B = np.asfortranarray(rng.standard_normal((L, H)) * np.ldexp(1.0, -r)[:, None])      # P[m, :] ~ 2^c_m
    A = np.asfortranarray(rng.standard_normal((M, H)) * np.ldexp(1.0, -c)[:, None])      # Q[l, :] ~ 2^r_l
    assert np.max(np.abs(Y)) > 2.0 ** 900 and np.min(np.abs(Y)) < 2.0 ** -900
    _check(G, ctx, num_sms, Y, B, A)


def test_subnormal_rows_and_entries(G, ctx, num_sms):
    L, M, H = 129, 161, 7
    rng = np.random.default_rng(5)
    Y, B, A = _inputs(rng, L, M, H)
    Y[[3, 70], :] = rng.standard_normal((2, M)) * 2.0 ** -1060       # whole rows in the subnormal range
    B[[3, 70], :] *= 2.0 ** 1000
    T = [10, 11, 90]
    Y[:, T] = rng.standard_normal((L, 3)) * 2.0 ** -1065             # subnormal columns: next to normal entries in each row
    A[T, :] *= 2.0 ** 1000
    assert np.all(np.abs(Y[3]) < 2.0 ** -1022) and np.any(np.abs(Y[5]) > 1e-10) and np.all(np.abs(Y[5, T]) < 2.0 ** -1022)
    _check(G, ctx, num_sms, Y, B, A)


def test_outputs_in_the_subnormal_range(G, ctx, num_sms):
    L, M, H = 129, 161, 7
    rng = np.random.default_rng(6)
    Y = np.asfortranarray(rng.standard_normal((L, M)) * 2.0 ** -530)
    B = np.asfortranarray(rng.standard_normal((L, H)) * 2.0 ** -530)
    A = np.asfortranarray(rng.standard_normal((M, H)) * 2.0 ** -535)
    assert np.all(np.abs(Y.T @ B) < 2.0 ** -1022)
    _check(G, ctx, num_sms, Y, B, A)


# ------------------------------------------------------------------------------------------- lifecycle of Y's digit planes
def test_reattach_synth_preprocess_and_chunked_attach(G, ctx, num_sms, monkeypatch):
    L, M, H = 129, 161, 9
    rng = np.random.default_rng(7)
    Y1, B, A = _inputs(rng, L, M, H)
    Y2, _, _ = _inputs(rng, L, M, H)
    _check(G, ctx, num_sms, Y1, B, A)
    _check(G, ctx, num_sms, Y2, B, A)                            # same shape: buffers kept, digits rebuilt
    ctx.synth(L, M, rank=4, noise=0.1, seed=3)
    _check(G, ctx, num_sms, ctx.download_Y(), B, A, attach=False)
    Yp = np.asfortranarray(rng.standard_normal((L, M)))        # no constant row: every row kept, scaled in place
    ctx.attach(Yp)
    ctx.preprocess(1.0)
    assert ctx.L == L
    _check(G, ctx, num_sms, ctx.download_Y(), B, A, attach=False)
    Y3 = Yp.copy()
    Y3[[5, 40], :] = 1.0                                         # constant rows are removed
    ctx.attach(Y3)
    rows = ctx.preprocess(1.0)
    assert ctx.L == L - 2 and 6 not in rows and 41 not in rows
    _check(G, ctx, num_sms, ctx.download_Y(), np.asfortranarray(B[:L - 2]), A, attach=False)
    # chunked asynchronous upload: 1 MB chunks of 896 columns
    Y4, B4, A4 = _inputs(rng, L, 4000, H)
    monkeypatch.setenv("VBMF_B200_ATTACH_CHUNK_MB", "1")
    _check(G, ctx, num_sms, Y4, B4, A4)
    monkeypatch.delenv("VBMF_B200_ATTACH_CHUNK_MB")
    _check(G, ctx, num_sms, Y4[:, ::-1].copy(order="F"), B4, A4)


# ------------------------------------------------------------------------------------------- non-finite inputs
@pytest.mark.parametrize("L,M", [(129, 161), (2000, 3001)])
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_nonfinite_inputs_give_nan_exactly_where_they_reach(G, ctx, num_sms, L, M, bad):
    H = 7
    rng = np.random.default_rng(8)
    Y, B, A = _inputs(rng, L, M, H)
    Y[L - 3, 5] = bad
    Y[7, M - 2] = bad
    B[L // 3, 2] = bad
    A[M - 1, 4] = bad
    ctx.attach(Y)
    P, Q = ctx.gemm_YtB(B), ctx.gemm_YA(A)
    Pmask = np.zeros((M, H), bool)
    Pmask[~np.all(np.isfinite(Y), axis=0), :] = True
    Pmask[:, ~np.all(np.isfinite(B), axis=0)] = True
    Qmask = np.zeros((L, H), bool)
    Qmask[~np.all(np.isfinite(Y), axis=1), :] = True
    Qmask[:, ~np.all(np.isfinite(A), axis=0)] = True
    assert np.array_equal(np.isnan(P), Pmask) and np.array_equal(np.isnan(Q), Qmask)
    assert not np.any(np.isinf(P)) and not np.any(np.isinf(Q))
    _check(G, ctx, num_sms, Y, B, A, attach=False)             # the rest is the model on the inputs with 0 in place


def _with_gemm(path, fn):
    old = os.environ.get("VBMF_B200_GEMM")
    try:
        if path == "dmma":
            os.environ["VBMF_B200_GEMM"] = "dmma"
        else:
            os.environ.pop("VBMF_B200_GEMM", None)
        return fn()
    finally:
        if old is None:
            os.environ.pop("VBMF_B200_GEMM", None)
        else:
            os.environ["VBMF_B200_GEMM"] = old


def test_dense_solver_with_a_nan_in_Y_matches_the_fp64_path(G):
    from tests.helpers import synth
    L, M, H = 200, 300, 64
    Y = np.asfortranarray(synth(L, M, 8, seed=2))
    Y[17, 33] = np.nan
    p0 = G.vb.vbmf_init(Y, H, rng=np.random.default_rng(9))

    def run():
        c = G.vb.Context(device=0)
        q = G.vb.copy(p0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            G.vb.vbmf_(Y, q, 20, eps=1e-9, est_covs=True, est_var=True, ctx=c)
        c.close()
        return q

    qi, qd = _with_gemm("int8", run), _with_gemm("dmma", run)
    assert not np.all(np.isfinite(qi.BHat)) and not np.all(np.isfinite(qi.AHat))
    for f in ("AHat", "BHat"):
        assert np.array_equal(np.isfinite(getattr(qi, f)), np.isfinite(getattr(qd, f))), f
    assert qi.iterations == qd.iterations and getattr(qi, "failed", False) == getattr(qd, "failed", False)


# ------------------------------------------------------------------------------------------- spectral norm at extreme scales
def _dense_problem(G):
    from tests.helpers import synth
    L, M, H = 60, 80, 4
    Y = np.asfortranarray(synth(L, M, 3, seed=5))
    return Y, G.vb.vbmf_init(Y, H, rng=np.random.default_rng(10))


def _run_scaled(G, ctx, Y, p0, j, niter=200, eps=1e-5):
    s = 4.0 ** j
    q = G.vb.copy(p0)
    q.BHat = q.BHat * s
    q.SigmaB, q.CB, q.invCB = q.SigmaB * s * s, q.CB * s * s, q.invCB / (s * s)
    q.sigma2 = q.sigma2 * s * s
    G.vb.vbmf_(np.asfortranarray(Y * s), q, niter, eps=eps, est_covs=True, est_var=True, ctx=ctx)
    return q


@pytest.mark.parametrize("j", [-75, -70, -40, 40, 70, 75])
def test_dense_solver_is_scale_equivariant(G, ctx, j):
    """Y -> sY, BHat0 -> s BHat0, SigmaB0 / CB -> s^2, sigma2 -> s^2 with s = 4^j: every dense update is equivariant
    (AHat, SigmaA, CA, d unchanged; BHat scales by s; SigmaB, CB, sigma2 by s^2).  Powers of two scale exactly, and s^2 a
    power of four keeps the square roots of the equilibration exact.  At |j| >= 70 the Grams D'D and BHat'BHat of the
    convergence test pass 1e+-80, where an unscaled Sturm recurrence of the spectral norm overflows or underflows."""
    Y, p0 = _dense_problem(G)
    ref = _run_scaled(G, ctx, Y, p0, 0)
    q = _run_scaled(G, ctx, Y, p0, j)
    s = 4.0 ** j
    assert 5 < ref.iterations < 200
    assert q.iterations == ref.iterations and q.d == ref.d
    for f, k in (("AHat", 0), ("SigmaA", 0), ("CA", 0), ("BHat", 1), ("SigmaB", 2), ("CB", 2)):
        assert np.array_equal(getattr(q, f) / s ** k, getattr(ref, f)), f
    assert q.sigma2 / (s * s) == ref.sigma2


@pytest.mark.parametrize("H,est_covs,seed", [(1, True, 2), (2, False, 1)])
def test_bitwise_fixed_point_stops_the_loop_with_d_zero(G, ctx, H, est_covs, seed):
    # Seeded problems whose own GPU iteration reaches a bitwise fixed point of BHat (found by running at eps = 0 until the
    # loop stopped with d == 0).  At the first K with BHat_K == BHat_{K-1}, D'D is exactly zero, its spectral norm must be
    # exactly 0, d = 0 / norm(Bold) = 0, and the reference's `d > eps` with eps = 0 ends the loop there.
    from tests.helpers import synth
    L, M = 10, 20
    Y = np.asfortranarray(synth(L, M, H, seed=seed))
    p0 = G.vb.vbmf_init(Y, H, rng=np.random.default_rng(seed))

    def run(niter):
        q = G.vb.copy(p0)
        G.vb.vbmf_(Y, q, niter, eps=0.0, est_covs=est_covs, ctx=ctx)
        return q

    full = run(2000)
    K = full.iterations
    assert K < 2000 and full.d == 0.0
    before, at = run(K - 2), run(K - 1)
    assert not np.array_equal(before.BHat, at.BHat) and at.d > 0.0       # BHat still moved at iteration K - 1
    last = run(K)
    assert np.array_equal(last.BHat, at.BHat) and last.d == 0.0           # and repeats bit for bit at K
    assert last.iterations == K and np.array_equal(full.BHat, last.BHat)


def test_zero_gram_stops_the_loop_like_the_reference(G, ctx):
    # Y = 0: BHat is exactly 0 from the first update on, so at the second iteration D = BHat - Bold = 0 and norm(Bold) = 0.
    # The reference's d = norm(D) / norm(Bold) is then NaN and `d > eps` ends the loop; the spectral norm of the zero Gram
    # must be exactly 0 for the device loop to stop there too.
    from oracle import vbmf_oracle as vo
    L, M, H = 10, 20, 2
    Y = np.zeros((L, M), order="F")
    p = vo.vbmf_init(Y, H, rng=np.random.default_rng(11))
    q = G.to_gpu_params(p)
    _, it, d = vo.vbmf_run(Y, p, 50, eps=0.0)
    G.vb.vbmf_(Y, q, 50, eps=0.0, ctx=ctx)
    assert it == 2 and q.iterations == it
    assert np.isnan(d) and np.isnan(q.d)
