"""Batched lowerBound / lowerBoundTrimmed (vbmf_b200_batched_lower_bound, BatchedVbls.lower_bound, lowerBound_batched,
lowerBoundTrimmed_batched) against the oracle and against the single-solver lowerBound, one problem at a time."""
import numpy as np
import pytest

from oracle import vbmf_oracle as vo
from tests.helpers import synth

pytestmark = pytest.mark.gpu
TOL = 1e-10
TOL_SINGLE = 1e-12
HUGE_TRIM = 1e300          # above every |AHat|: nothing is kept


@pytest.fixture(scope="module")
def G():
    from tests import gpu_helpers
    return gpu_helpers


@pytest.fixture(scope="module")
def ctx(G):
    c = G.vb.Context(device=0)
    yield c
    c.close()


def _state(kind, L, M, H, seed, H0=None, M0=None, niter=3, full_cov=False):
    """An oracle state after `niter` iterations of the kind's own loop from its initialiser (default hyper-priors 1e-10)."""
    rng = np.random.default_rng(seed)
    Y = 10.0 * synth(L, M, max(1, min(3, H)), seed=seed)
    if kind == "sparse":
        p = vo.vbmf_sparse_init(Y, H, rng=rng)
        run = vo.vbmf_sparse_run
    elif kind == "dual":
        p = vo.vbmf_dual_init(Y, H, H - 1 if H0 is None else H0, rng=rng)
        run = vo.vbmf_dual_run
    else:
        p = vo.vbmf_trial_init(Y, H, max(H - 2, 0) if H0 is None else H0, M // 2 if M0 is None else M0, rng=rng)
        run = vo.vbmf_trial_run
    if niter:   # the hyper-priors stay at their 1e-10 defaults (est_priors would turn an empty group's into NaN)
        run(Y, p, niter, eps=0.0, full_cov=full_cov, **({} if kind == "sparse" else {"est_priors": False}))
    return np.asfortranarray(Y), p


def _oracle(kind, Y, p, trim):
    fn = {"sparse": (vo.sparse_lowerBound, vo.sparse_lowerBoundTrimmed), "dual": (vo.dual_lowerBound, vo.dual_lowerBoundTrimmed),
          "trial": (vo.trial_lowerBound, vo.trial_lowerBoundTrimmed)}[kind]
    return fn[0](Y, p) if trim is None else fn[1](Y, p, trim)


def _single(G, ctx, Y, q, trim):
    return G.vb.lowerBound(Y, q, ctx=ctx) if trim is None else G.vb.lowerBoundTrimmed(Y, q, trim, ctx=ctx)


def _batched(G, ctx, Ys, qs, trim):
    return G.vb.lowerBound_batched(Ys, qs, ctx=ctx) if trim is None else G.vb.lowerBoundTrimmed_batched(Ys, qs, trim, ctx=ctx)


def _close(a, b, tol):
    if not np.isfinite(b):
        return a == b or (np.isnan(a) and np.isnan(b))
    return abs(a - b) <= tol * abs(b)


def _check(G, ctx, kind, problems, trims=(None, 0.1, HUGE_TRIM)):
    """Every problem of one batch against the oracle (TOL) and the single-solver path (TOL_SINGLE)."""
    Ys = [Y for Y, _ in problems]
    qs = [G.to_gpu_params(p) for _, p in problems]
    for trim in trims:
        got = _batched(G, ctx, Ys, qs, trim)
        assert got.dtype == np.float64 and got.shape == (len(problems),)
        for i, (Y, p) in enumerate(problems):
            want = _oracle(kind, Y, p, trim)
            assert _close(got[i], want, TOL), (kind, trim, i, got[i], want)
            one = _single(G, ctx, Y, G.to_gpu_params(p), trim)
            assert _close(got[i], one, TOL_SINGLE), (kind, trim, i, got[i], one)
    return Ys, qs


SHAPES = [  # L, H, Ms: odd H, H = 1, H = 64, L = 1, M = 1
    (30, 5, [1, 9, 40]),
    (25, 1, [1, 17]),
    (38, 64, [1, 70, 300]),
    (1, 3, [1, 6, 20]),
]


@pytest.mark.parametrize("kind", ["sparse", "dual", "trial"])
@pytest.mark.parametrize("L,H,Ms", SHAPES)
def test_every_kind_against_oracle(G, ctx, kind, L, H, Ms):
    _check(G, ctx, kind, [_state(kind, L, M, H, seed=100 + 7 * i + M) for i, M in enumerate(Ms)])


@pytest.mark.parametrize("H0", [0, 6])
def test_dual_empty_groups(G, ctx, H0):
    _check(G, ctx, "dual", [_state("dual", 24, M, 6, seed=200 + M, H0=H0) for M in (1, 11, 50)])


def test_trial_row_splits(G, ctx):
    M = 40
    _check(G, ctx, "trial", [_state("trial", 24, M, 6, seed=300 + M0, H0=3, M0=M0) for M0 in (0, M, 13)])


def test_entropy_q7_in_one_batch(G, ctx):
    """normalEntropy(kron(SigmaB, I_L)) at odd L: det(SigmaB)^L underflowing, overflowing, negative, and a pivoting
    indefinite SigmaB, next to ordinary problems; every value as the oracle's and the ordinary ones unaffected."""
    L, H = 41, 5
    rng = np.random.default_rng(5)
    probs = [_state("sparse", L, M, H, seed=400 + M) for M in (3, 20, 33, 8, 12, 27)]
    probs[1][1].SigmaB = np.eye(H) * 1e-3                     # L*log(det) ~ -1416: the running product underflows
    probs[2][1].SigmaB = np.eye(H) * 1e3                      # ~ +1416: overflows, positive sign -> +Inf
    probs[3][1].SigmaB = np.diag([1.0, 0.9, -1.1, 0.8, 1.2])  # negative determinant at odd L -> log(eps(0.0))
    S = rng.standard_normal((H, H))
    probs[4][1].SigmaB = 0.3 * (S + S.T)                      # indefinite, partial pivoting swaps rows
    probs[5][1].SigmaB = 0.9 * np.eye(H) + 0.01 * (S + S.T)   # finite log-determinant
    alone = [_batched(G, ctx, [Y], [G.to_gpu_params(p)], None)[0] for Y, p in probs]
    _check(G, ctx, "sparse", probs, trims=(None, 0.1))
    got = _batched(G, ctx, [Y for Y, _ in probs], [G.to_gpu_params(p) for _, p in probs], None)
    assert np.isinf(got[2]) and got[2] > 0
    assert [v.hex() for v in got] == [v.hex() for v in alone]


def test_after_batched_vbls_musk2_shaped(G, ctx):
    """BatchedVbls.run(20, full_cov) then .lower_bound() / .lower_bound(0.1) on Musk2-shaped dual bags (L = 166, H = 20),
    against oracle vbls followed by lowerBound on every problem."""
    L, H, H0 = 166, 20, 19
    rng = np.random.default_rng(2026)
    B = [np.asfortranarray(rng.standard_normal((L, H))) for _ in range(2)]
    SB = [np.diag(rng.uniform(1e-3, 1e-2, H)) for _ in range(2)]
    Ys, ps = [], []
    for M in (1, 7, 300, 1044):
        Y = np.asfortranarray(10.0 * (rng.standard_normal((L, 3)) @ rng.standard_normal((3, M)) + 0.1 * rng.standard_normal((L, M))))
        for c in range(2):
            p = vo.vbmf_dual_init(Y, H, H0, rng=rng)
            p.BHat, p.SigmaB, p.sigmaHat = B[c].copy(), SB[c].copy(), 0.7
            Ys.append(Y)
            ps.append(p)
    qs = [G.to_gpu_params(p) for p in ps]
    batch = G.vb.BatchedVbls(Ys, qs, ctx=ctx, yhat=True)
    batch.run(20, full_cov=True)
    lb, lbt = batch.lower_bound(), batch.lower_bound(0.1)
    batch.readback()
    for i, (Y, p) in enumerate(zip(Ys, ps)):
        vo.vbls(Y, p, 20, full_cov=True)
        assert _close(lb[i], vo.dual_lowerBound(Y, p), TOL), (i, lb[i], vo.dual_lowerBound(Y, p))
        assert _close(lbt[i], vo.dual_lowerBoundTrimmed(Y, p, 0.1), TOL), i
        assert _close(lb[i], G.vb.lowerBound(Y, qs[i], ctx=ctx), TOL_SINGLE), i
        assert _close(lbt[i], G.vb.lowerBoundTrimmed(Y, qs[i], 0.1, ctx=ctx), TOL_SINGLE), i


def test_large_problem_split_over_ctas(G, ctx):
    """1e5 columns (many CTAs on one problem): oracle TOL, single-solver agreement, and bit-identical alone, inside a mixed
    batch and across runs."""
    big = _state("dual", 20, 100000, 8, seed=500, niter=0)
    small = [_state("dual", 20, M, 8, seed=510 + M) for M in (1, 5000, 333)]
    for trim in (None, 0.1):
        Yb, qb = [big[0]], [G.to_gpu_params(big[1])]
        alone = _batched(G, ctx, Yb, qb, trim)
        again = _batched(G, ctx, Yb, qb, trim)
        mixed = _batched(G, ctx, [small[0][0], big[0], small[1][0], small[2][0]],
                         [G.to_gpu_params(small[0][1]), qb[0], G.to_gpu_params(small[1][1]), G.to_gpu_params(small[2][1])], trim)
        assert alone[0].hex() == again[0].hex() == mixed[1].hex()
        assert _close(alone[0], _oracle("dual", big[0], big[1], trim), TOL)
        assert _close(alone[0], _single(G, ctx, big[0], G.to_gpu_params(big[1]), trim), TOL_SINGLE)
        for j, k in ((0, 0), (2, 1), (3, 2)):
            assert _close(mixed[j], _oracle("dual", small[k][0], small[k][1], trim), TOL)


def test_bad_state_is_nan_for_its_problem_only(G, ctx):
    probs = [_state("dual", 24, M, 6, seed=600 + M) for M in (4, 9, 15)]
    Ys = [Y for Y, _ in probs]
    clean = _batched(G, ctx, Ys, [G.to_gpu_params(p) for _, p in probs], None)
    qs = [G.to_gpu_params(p) for _, p in probs]
    qs[1].beta[3] = -1.0
    got = _batched(G, ctx, Ys, qs, None)
    assert np.isnan(got[1]) and np.isfinite(got[[0, 2]]).all()
    assert got[0].hex() == clean[0].hex() and got[2].hex() == clean[2].hex()


def test_arena_regrowth(G, ctx):
    small = [_state("sparse", 20, M, 8, seed=700 + M) for M in (3, 30)]
    big = _state("sparse", 20, 60000, 8, seed=710, niter=0)
    Ys, qs = [Y for Y, _ in small], [G.to_gpu_params(p) for _, p in small]
    first = _batched(G, ctx, Ys, qs, None)
    large = _batched(G, ctx, [big[0]] + Ys, [G.to_gpu_params(big[1])] + qs, None)
    last = _batched(G, ctx, Ys, qs, None)
    assert [v.hex() for v in first] == [v.hex() for v in last] == [v.hex() for v in large[1:]]
    assert _close(large[0], vo.sparse_lowerBound(big[0], big[1]), TOL)


def test_resident_y_and_live_solver_untouched(G, ctx):
    """A batched call between two steps of a live solver on an attached Y changes neither trYTY nor the solver's results."""
    Y0, p0 = _state("sparse", 30, 200, 6, seed=800)
    c = G.vb.Context(device=0)
    try:
        c.attach(Y0, force=True)
        tr = c.trYTY()
        s = G.vb.Solver(c, G.to_gpu_params(p0))
        try:
            s.upload(G.to_gpu_params(p0))
            before = s.lower_bound()
            probs = [_state("sparse", 30, M, 6, seed=810 + M) for M in (2, 90)]
            _batched(G, c, [Y for Y, _ in probs], [G.to_gpu_params(p) for _, p in probs], 0.1)
            assert s.lower_bound() == before
            assert c.trYTY() == tr
            s.run(2, eps=0.0)
            q = G.to_gpu_params(p0)
            s.download(q)
            ref = G.vb.Context(device=0)
            try:
                ref.attach(Y0, force=True)
                t = G.vb.Solver(ref, G.to_gpu_params(p0))
                t.upload(G.to_gpu_params(p0))
                t.run(2, eps=0.0)
                r = G.to_gpu_params(p0)
                t.download(r)
                t.close()
            finally:
                ref.close()
            assert np.array_equal(q.BHat, r.BHat) and np.array_equal(q.AHat, r.AHat)
        finally:
            s.close()
    finally:
        c.close()


def test_refusals(G, ctx):
    Y, p = _state("dual", 12, 10, 4, seed=900)
    Ys, q = [Y], G.to_gpu_params(p)
    with pytest.raises(G.vb.VBMFError, match="no lowerBound"):
        G.vb.lowerBound_batched([Y], [G.vb.vbmf_init(Y, 2)], ctx=ctx)
    Ys2, ps2 = _state("sparse", 12, 10, 4, seed=901)
    with pytest.raises(G.vb.VBMFError):
        G.vb.lowerBound_batched([Y, Ys2], [q, G.to_gpu_params(ps2)], ctx=ctx)                     # mixed kinds
    for other in (_state("dual", 13, 10, 4, seed=902), _state("dual", 12, 10, 5, seed=903),
                  _state("dual", 12, 10, 4, seed=904, H0=1)):                                     # L, H, H0 differ
        with pytest.raises(G.vb.VBMFError):
            G.vb.lowerBound_batched([Y, other[0]], [q, G.to_gpu_params(other[1])], ctx=ctx)
    Yh, ph = _state("sparse", 70, 3, 65, seed=905, niter=0)
    with pytest.raises(G.vb.VBMFError, match="H <= 64"):
        G.vb.lowerBoundTrimmed_batched([Yh], [G.to_gpu_params(ph)], ctx=ctx)
    qm = G.to_gpu_params(p)
    qm.ATVecHat = qm.ATVecHat + 1.0
    with pytest.raises(G.vb.VBMFError, match="disagree"):
        G.vb.lowerBound_batched(Ys, [qm], ctx=ctx)
    m = G.vb.MultiContext(devices=[0])
    try:
        with pytest.raises(G.vb.VBMFError, match="one device"):
            G.vb.lowerBound_batched(Ys, [q], ctx=m)
        with pytest.raises(G.vb.VBMFError, match="one device"):
            G.vb.lowerBoundTrimmed_batched(Ys, [q], ctx=m)
    finally:
        m.close()
    assert G.vb.lowerBound_batched([], [], ctx=ctx).shape == (0,)
