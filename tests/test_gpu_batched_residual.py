"""Batched residual norms norm(Y - BHat*AHat') (vbmf_b200_batched_residual_norm, BatchedVbls.residual_norm,
residual_norm_batched) against NumPy on the host, against mil.classify_bags, and for batch invariance, extreme scales,
non-finite values, side effects and refusals."""
import ctypes as C

import numpy as np
import pytest

from tests.helpers import synth

pytestmark = pytest.mark.gpu
TOL = 1e-12
KINDS = ("dense", "sparse", "dual", "trial")


@pytest.fixture(scope="module")
def vb():
    from tests import gpu_helpers
    return gpu_helpers.vb


@pytest.fixture(scope="module")
def ctx(vb):
    c = vb.Context(device=0)
    yield c
    c.close()


def _params(vb, kind, Y, H, rng):
    """A state of `kind` for Y with random factors: only L, M, H, BHat and AHat take part in the norm."""
    L, M = Y.shape
    if kind == "dense":
        p = vb.vbmf_init(Y, H, rng=rng)
    elif kind == "sparse":
        p = vb.vbmf_sparse_init(Y, H, rng=rng)
    elif kind == "dual":
        p = vb.vbmf_dual_init(Y, H, max(H - 1, 0), rng=rng)
    else:
        p = vb.vbmf_trial_init(Y, H, max(H - 2, 0), M // 2, rng=rng)
    p.BHat = np.asfortranarray(rng.standard_normal((L, H)))
    p.AHat = np.asfortranarray(0.3 * rng.standard_normal((M, H)))
    return p


def _batch(vb, kind, L, H, Ms, seed):
    rng = np.random.default_rng(seed)
    Ys = [np.asfortranarray(rng.standard_normal((L, M))) for M in Ms]
    return Ys, [_params(vb, kind, Y, H, rng) for Y in Ys]


def _host(Y, p, norm):
    return float(np.linalg.norm(Y - np.asarray(p.BHat) @ np.asarray(p.AHat).T, 2 if norm == "spectral" else "fro"))


def _check(vb, ctx, Ys, ps, norms=("spectral", "frobenius")):
    for norm in norms:
        got = vb.residual_norm_batched(Ys, ps, norm=norm, ctx=ctx)
        assert got.dtype == np.float64 and got.shape == (len(ps),)
        for i, (Y, p) in enumerate(zip(Ys, ps)):
            want = _host(Y, p, norm)
            assert abs(got[i] - want) <= TOL * want, (norm, i, Y.shape, got[i], want)


def _bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64)


# ---- values ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("L,H,Ms", [(30, 7, [20, 30, 45, 1, 64]),     # M < L, M = L, M > L, M = 1, two Gram tiles
                                     (1, 3, [1, 9, 4]),                 # L = 1
                                     (38, 20, [5, 40, 17]),             # the c2 shape
                                     (12, 1, [3, 100])])                # H = 1
def test_all_kinds_match_host(vb, ctx, kind, L, H, Ms):
    Ys, ps = _batch(vb, kind, L, H, Ms, seed=L * 100 + H)
    _check(vb, ctx, Ys, ps)


@pytest.mark.parametrize("L,Ms", [(168, [168, 500, 3]),      # n = 168: the largest Gram in shared memory
                                  (169, [169, 400]),         # n = 169: the smallest one in global memory
                                  (300, [400, 250, 301])])   # n = 250..300, global memory
def test_shared_and_global_gram(vb, ctx, L, Ms):
    Ys, ps = _batch(vb, "dual", L, 20, Ms, seed=L)
    _check(vb, ctx, Ys, ps)


def test_musk2_shape(vb, ctx):
    """tools/batched/large_bags.make_batch: 100 bags of 1..1044 columns at L = 166 against two class models."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "batched"))
    from large_bags import make_batch
    Ys, ps = make_batch(vb)
    assert max(Y.shape[1] for Y in Ys) == 1044
    _check(vb, ctx, Ys, ps)


def test_c2_sized_batch(vb, ctx):
    rng = np.random.default_rng(38)
    Ms = rng.integers(5, 41, 548)
    Ys = [np.asfortranarray(10.0 * synth(38, int(M), 3, seed=i)) for i, M in enumerate(Ms)]
    ps = [_params(vb, "dual", Y, 20, rng) for Y in Ys for _ in range(2)]
    Ys = [Y for Y in Ys for _ in range(2)]
    _check(vb, ctx, Ys, ps)


# ---- the MIL classifiers ----------------------------------------------------------------------------------------------------
def _class_models(vb, kind, L, H, seed):
    rng = np.random.default_rng(seed)
    out = []
    for c in range(2):
        Yt = 10.0 * synth(L, 60, 3, seed=seed + c)
        p = vb.vbmf_dual_init(Yt, H, H - 1, rng=rng) if kind == "dual" else vb.vbmf_init(Yt, H, rng=rng)
        p.BHat = np.asfortranarray(rng.standard_normal((L, H)))
        p.SigmaB = np.asfortranarray(np.diag(rng.uniform(1e-3, 1e-2, H)))
        if kind == "dual":
            p.sigmaHat = 0.7
        out.append(p)
    return out


@pytest.mark.parametrize("class_alg", ["dual", "vbls"])
def test_matches_classify_bags(vb, ctx, class_alg):
    """BatchedVbls.run + residual_norm reproduces mil.classify_bags: the same errors to 1e-12 and the same labels."""
    L, H = 38, 12
    kind = "dual" if class_alg == "dual" else "dense"
    res = _class_models(vb, kind, L, H, seed=5)
    rng = np.random.default_rng(11)
    Ys = [np.asfortranarray(10.0 * synth(L, int(M), 3, seed=100 + i) + rng.standard_normal((L, int(M))))
          for i, M in enumerate(rng.integers(1, 60, 40))]
    labels, e0, e1 = vb.mil.classify_bags(res[0], res[1], Ys, class_alg=class_alg, ctx=ctx, rng=np.random.default_rng(3))
    niter, full_cov = (20, True) if class_alg == "dual" else (150, False)
    rng = np.random.default_rng(3)
    errs = []
    for r in res:
        ps = [vb.mil.copy_vbmf_params(Y, r, rng=rng) for Y in Ys]
        batch = vb.BatchedVbls(Ys, ps, ctx=ctx, yhat=False)
        batch.run(niter, full_cov=full_cov)
        e = batch.residual_norm()
        errs.append(e / np.array([Y.size for Y in Ys]) if class_alg == "dual" else e)
    for got, want in zip(errs, (e0, e1)):
        assert np.all(np.abs(got - want) <= TOL * np.abs(want)), np.max(np.abs(got - want) / np.abs(want))
    mine = np.where(errs[0] < errs[1], 0, 1) if class_alg == "dual" else np.where(errs[0] > errs[1], 1, 0)
    assert np.array_equal(mine, labels)


# ---- batch invariance ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("norm", ["spectral", "frobenius"])
@pytest.mark.parametrize("L,Ms", [(50, [3, 60, 200, 50, 17, 1]), (200, [150, 300, 7])])
def test_batch_invariance(vb, ctx, norm, L, Ms):
    Ys, ps = _batch(vb, "sparse", L, 9, Ms, seed=7)
    full = vb.residual_norm_batched(Ys, ps, norm=norm, ctx=ctx)
    alone = np.array([vb.residual_norm_batched([Y], [p], norm=norm, ctx=ctx)[0] for Y, p in zip(Ys, ps)])
    perm = np.random.default_rng(1).permutation(len(ps))
    permuted = vb.residual_norm_batched([Ys[i] for i in perm], [ps[i] for i in perm], norm=norm, ctx=ctx)
    again = vb.residual_norm_batched(Ys, ps, norm=norm, ctx=ctx)
    assert np.array_equal(_bits(full), _bits(alone))
    assert np.array_equal(_bits(full[perm]), _bits(permuted))
    assert np.array_equal(_bits(full), _bits(again))


# ---- scale and non-finite values ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [500, -500, 600, -600])
def test_power_of_two_scaling(vb, ctx, s):
    """Y and BHat times 2^s: the residual is scaled exactly, and so is its norm, bit for bit."""
    Ys, ps = _batch(vb, "dual", 40, 6, [10, 40, 90], seed=3)
    base = {n: vb.residual_norm_batched(Ys, ps, norm=n, ctx=ctx) for n in ("spectral", "frobenius")}
    Ys2 = [np.asfortranarray(np.ldexp(Y, s)) for Y in Ys]
    for p in ps:
        p.BHat = np.asfortranarray(np.ldexp(p.BHat, s))
    for n in ("spectral", "frobenius"):
        got = vb.residual_norm_batched(Ys2, ps, norm=n, ctx=ctx)
        assert np.all(np.isfinite(got)) and np.all(got > 0)
        assert np.array_equal(_bits(got), _bits(np.ldexp(base[n], s))), (n, got, np.ldexp(base[n], s))


@pytest.mark.parametrize("bad", [np.nan, np.inf])
def test_non_finite_stays_in_its_problem(vb, ctx, bad):
    Ys, ps = _batch(vb, "sparse", 30, 5, [12, 40, 7, 200], seed=9)
    ref = {n: vb.residual_norm_batched(Ys, ps, norm=n, ctx=ctx) for n in ("spectral", "frobenius")}
    Ys[1] = Ys[1].copy(order="F")
    Ys[1][3, 5] = bad
    Ys[3] = Ys[3].copy(order="F")
    Ys[3][29, 150] = bad                    # M > L: the RR' orientation
    for n in ("spectral", "frobenius"):
        got = vb.residual_norm_batched(Ys, ps, norm=n, ctx=ctx)
        if n == "spectral" or np.isnan(bad):
            assert np.isnan(got[1]) and np.isnan(got[3])
        else:
            assert got[1] == np.inf and got[3] == np.inf
        assert np.array_equal(_bits(got[[0, 2]]), _bits(ref[n][[0, 2]]))


def test_zero_residual_is_exactly_zero(vb, ctx):
    Ys, ps = _batch(vb, "dense", 20, 4, [5, 20, 60], seed=2)
    for i, p in enumerate(ps):
        p.AHat = np.asfortranarray(np.zeros_like(p.AHat))
        Ys[i] = np.asfortranarray(np.zeros_like(Ys[i]))
    for n in ("spectral", "frobenius"):
        assert np.array_equal(vb.residual_norm_batched(Ys, ps, norm=n, ctx=ctx), np.zeros(3))


# ---- side effects -------------------------------------------------------------------------------------------------------------
def _snapshot(p):
    return {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in vars(p).items()}


@pytest.mark.parametrize("kind", KINDS)
def test_states_are_left_unchanged(vb, ctx, kind):
    Ys, ps = _batch(vb, kind, 25, 5, [4, 25, 70], seed=4)
    batch = vb.BatchedVbls(Ys, ps, ctx=ctx, yhat=False)
    before = [_snapshot(p) for p in ps]
    raw = [C.string_at(C.addressof(st), C.sizeof(st)) for st in batch.structs]
    for n in ("spectral", "frobenius"):
        batch.residual_norm(n)
    assert raw == [C.string_at(C.addressof(st), C.sizeof(st)) for st in batch.structs]
    for b, p in zip(before, ps):
        after = _snapshot(p)
        assert b.keys() == after.keys()
        for k in b:
            if isinstance(b[k], np.ndarray):
                assert b[k].tobytes() == after[k].tobytes(), k
            else:
                assert b[k] == after[k] or (b[k] != b[k] and after[k] != after[k]), k


def test_resident_y_and_live_solver_untouched(vb, ctx):
    """A solver on the context's resident Y runs on to the same bits with a batched residual norm in between."""
    Y = np.asfortranarray(synth(200, 3000, 5, seed=21))
    Ys, ps = _batch(vb, "dual", 166, 20, [1044, 300, 9], seed=8)    # grows the staging arena
    out = []
    for between in (False, True):
        ctx.attach(Y, force=True)
        q = vb.vbmf_sparse_init(Y, 8, rng=np.random.default_rng(0))
        s = vb.Solver(ctx, q)
        try:
            s.upload(q)
            s.run(3, eps=0.0)
            if between:
                vb.residual_norm_batched(Ys, ps, ctx=ctx)
            s.run(3, eps=0.0)
            s.download(q, want_yhat=True)
        finally:
            s.close()
        out.append(q)
    for f in ("AHat", "BHat", "SigmaA", "SigmaB", "CA", "CB", "YHat"):
        assert np.array_equal(_bits(getattr(out[0], f)), _bits(getattr(out[1], f))), f
    assert out[0].sigmaHat == out[1].sigmaHat


# ---- refusals -----------------------------------------------------------------------------------------------------------------
def _raw(vb, ctx, kind, Ys, structs, mode=0):
    n = len(structs)
    ypt = (vb._lib.p_f64 * n)(*[Y.ctypes.data for Y in Ys])
    spt = (C.c_void_p * n)(*[C.addressof(st) if st is not None else None for st in structs])
    out = np.zeros(n)
    return ctx.lib.vbmf_b200_batched_residual_norm(ctx.h, kind, n, ypt, spt, mode, out.ctypes.data)


def _refused(vb, match, rc):
    assert rc == -1
    assert match in vb._lib.load().vbmf_b200_last_error().decode()


def test_refusals(vb, ctx):
    Ys, ps = _batch(vb, "sparse", 20, 4, [6, 9, 5], seed=12)
    batch = vb.BatchedVbls(Ys, ps, ctx=ctx, yhat=False)
    sts = batch.structs
    lib, out = ctx.lib, np.zeros(3)
    # NULL arguments and arrays
    _refused(vb, "NULL argument", lib.vbmf_b200_batched_residual_norm(None, 1, 3, batch.yp, batch.sp, 0, out.ctypes.data))
    _refused(vb, "NULL argument", lib.vbmf_b200_batched_residual_norm(ctx.h, 1, 3, None, batch.sp, 0, out.ctypes.data))
    _refused(vb, "NULL argument", lib.vbmf_b200_batched_residual_norm(ctx.h, 1, 3, batch.yp, None, 0, out.ctypes.data))
    _refused(vb, "NULL argument", lib.vbmf_b200_batched_residual_norm(ctx.h, 1, 3, batch.yp, batch.sp, 0, None))
    _refused(vb, "NULL problem 1", _raw(vb, ctx, 1, Ys, [sts[0], None, sts[2]]))
    yp = (vb._lib.p_f64 * 3)(Ys[0].ctypes.data, None, Ys[2].ctypes.data)
    _refused(vb, "NULL problem 1", lib.vbmf_b200_batched_residual_norm(ctx.h, 1, 3, yp, batch.sp, 0, out.ctypes.data))
    a = sts[2].AHat
    sts[2].AHat = None
    _refused(vb, "AHat of problem 2 is NULL", _raw(vb, ctx, 1, Ys, sts))
    sts[2].AHat = a
    # kind and norm mode
    _refused(vb, "unknown parameter kind 7", _raw(vb, ctx, 7, Ys, sts))
    _refused(vb, "unknown norm mode 2", _raw(vb, ctx, 1, Ys, sts, mode=2))
    with pytest.raises(vb.VBMFError, match="norm must be"):
        batch.residual_norm("nuclear")
    # batch rules
    sts[1].L = 21
    _refused(vb, "problem 1 has a different L or H", _raw(vb, ctx, 1, Ys, sts))
    sts[1].L = 20
    sts[2].H = 5
    _refused(vb, "problem 2 has a different L or H", _raw(vb, ctx, 1, Ys, sts))
    sts[2].H = 4
    sts[1].M = 0
    _refused(vb, "problem 1 has M < 1", _raw(vb, ctx, 1, Ys, sts))
    sts[0].M = sts[1].M = sts[2].M = 1 << 30          # refused before any Y is read
    _refused(vb, "more than 2^31 columns", _raw(vb, ctx, 1, Ys, sts))
    sts[0].M, sts[1].M, sts[2].M = 6, 9, 5
    assert np.all(batch.residual_norm() > 0)
    # the spectral norm needs min(L, M) <= 2048; the Frobenius norm does not
    Yb = np.asfortranarray(np.zeros((2049, 2049)))
    pb = _params(vb, "dense", Yb, 1, np.random.default_rng(0))
    with pytest.raises(vb.VBMFError, match=r"min\(L, M\) <= 2048"):
        vb.residual_norm_batched([Yb], [pb], ctx=ctx)
    got = vb.residual_norm_batched([Yb], [pb], norm="frobenius", ctx=ctx)[0]
    assert abs(got - _host(Yb, pb, "frobenius")) <= TOL * got
    # one device only
    m = vb.MultiContext(devices=[0])
    try:
        with pytest.raises(vb.VBMFError, match="MultiContext"):
            vb.residual_norm_batched(Ys, ps, ctx=m)
    finally:
        m.close()
