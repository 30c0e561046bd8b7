"""Batched vbls! on problems that do not fit one CTA's shared memory (the wide kernel, one thread-block cluster per
problem), against the oracle's vbls and against the one-CTA kernel for the problems that fit."""
import numpy as np
import pytest

from oracle import vbmf_oracle as vo
from tests.helpers import synth

pytestmark = pytest.mark.gpu
TOL = 1e-10


@pytest.fixture(scope="module")
def G():
    from tests import gpu_helpers
    return gpu_helpers


@pytest.fixture(scope="module")
def ctx(G):
    c = G.vb.Context(device=0)
    yield c
    c.close()


def _plan(G, kind, L, H, Ms, full_cov=True, diag_var=False):
    lib = G.vb._lib.load()
    M = np.asarray(Ms, dtype=np.int64)
    out = np.zeros(M.size, dtype=np.int32)
    kinds = {"dense": 0, "sparse": 1, "dual": 2, "trial": 3}
    G.vb._lib.check(lib.vbmf_b200_batched_plan(kinds[kind], L, H, int(full_cov), int(diag_var), M.size, M.ctypes.data, out.ctypes.data))
    return out


def _problem(kind, L, H, M, seed, rng, diag_var=False):
    Y = 10.0 * synth(L, M, 3, seed=seed)
    if kind == "sparse":
        p = vo.vbmf_sparse_init(Y, H, rng=rng)
    elif kind == "dense":
        p = vo.vbmf_init(Y, H, sigma2=0.9, rng=rng)
    elif kind == "trial":
        p = vo.vbmf_trial_init(Y, H, H - 2, M // 2, rng=rng)
        p.alpha01, p.beta01, p.alpha02, p.beta02, p.alpha03, p.beta03 = 0.3, 0.2, 0.7, 0.4, 1e-10, 1e-10
    else:
        p = vo.vbmf_dual_init(Y, H, H - 1, rng=rng)
    p.SigmaB = np.diag(rng.uniform(1e-3, 1e-2, H))
    if kind != "dense":
        p.sigmaHat = 0.7
        if diag_var:
            p.sigmaVecHat = rng.uniform(0.5, 2.0, L)
    return np.asfortranarray(Y), p


def _fields(kind, diag_var):
    if kind == "dense":
        return ["AHat", "SigmaA", "CA", "invCA", "sigma2"]
    f = ["AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "CA", "beta", "sigmaHat", "zeta"]
    if kind == "dual":
        f += ["A0Hat", "A1Hat", "CA0", "CA1", "beta0", "beta1", "alpha0", "alpha1"]
    if kind == "trial":
        f += ["A1Hat", "A2Hat", "A3Hat", "CA1", "CA2", "CA3", "beta1", "beta2", "beta3", "alpha1", "alpha2", "alpha3"]
    if diag_var:
        f += ["sigmaVecHat", "zetaVec"]
    return f


CASES = [  # kind, full_cov, diag_var, L, H, Ms
    ("dual", True, False, 166, 20, [1, 7, 300, 700, 1044]),
    ("dual", False, False, 166, 20, [1, 7, 300, 700, 1044]),
    ("sparse", True, True, 166, 20, [1, 7, 300, 700, 1044]),
    ("sparse", False, True, 166, 20, [7, 300, 1044]),
    ("trial", True, False, 166, 20, [7, 300, 700]),
    ("trial", False, True, 166, 20, [7, 700]),
    ("sparse", True, False, 38, 64, [2, 40, 200]),
    ("dual", True, True, 38, 64, [2, 40, 200]),
    ("sparse", False, False, 38, 64, [2, 40, 200]),
    ("dense", False, False, 166, 20, [1, 7, 300, 700, 1044]),
    ("dense", False, False, 166, 32, [7, 267, 600, 1044]),
]


@pytest.mark.parametrize("kind,full_cov,diag_var,L,H,Ms", CASES)
def test_large_bags_match_oracle(G, ctx, kind, full_cov, diag_var, L, H, Ms):
    rng = np.random.default_rng(L + H + len(Ms))
    niter = 8
    cs = _plan(G, kind, L, H, Ms, full_cov, diag_var)
    assert np.any(cs > 0)
    Ys, ps = zip(*[_problem(kind, L, H, M, 1000 + i, rng, diag_var) for i, M in enumerate(Ms)])
    qs = [G.to_gpu_params(p) for p in ps]
    G.vb.vbls_batched_(list(Ys), qs, niter, full_cov=full_cov, diag_var=diag_var, ctx=ctx, yhat=True, keep_blocks=full_cov)
    for Y, p, q in zip(Ys, ps, qs):
        vo.vbls(Y, p, niter, full_cov=full_cov, diag_var=diag_var)
        G.compare(q, p, TOL, _fields(kind, diag_var))
        assert G.rel(q.YHat, p.YHat) < TOL
        if full_cov:
            assert G.rel(q.SigmaATVec_blocks, p.SigmaATVec_blocks) < TOL


def test_every_cluster_size_matches_oracle(G, ctx):
    """One batch with problems of cluster size 1, 2, 4 and 8 (L = 38, H = 64: two columns do not fit one CTA)."""
    L, H, Ms = 38, 64, [40, 100, 200, 600]
    assert _plan(G, "sparse", L, H, Ms).tolist() == [1, 2, 4, 8]
    rng = np.random.default_rng(4)
    Ys, ps = zip(*[_problem("sparse", L, H, M, 50 + i, rng) for i, M in enumerate(Ms)])
    qs = [G.to_gpu_params(p) for p in ps]
    G.vb.vbls_batched_(list(Ys), qs, 5, full_cov=True, ctx=ctx, keep_blocks=True)
    for Y, p, q in zip(Ys, ps, qs):
        vo.vbls(Y, p, 5, full_cov=True)
        G.compare(q, p, TOL, _fields("sparse", False))
        assert G.rel(q.YHat, p.YHat) < TOL and G.rel(q.SigmaATVec_blocks, p.SigmaATVec_blocks) < TOL


def _c2_small(G, rng, n=24, kind="dual", diag_var=False):
    return [_problem(kind, 166, 20, int(rng.integers(5, 41)), 300 + b, rng, diag_var) for b in range(n)]


def _snap(q, kind="dual"):
    return {f: np.array(getattr(q, f), dtype=np.float64, copy=True) for f in _fields(kind, False) + ["YHat"]}


def test_mixed_batch_keeps_small_bags_on_the_one_cta_kernel(G, ctx):
    rng = np.random.default_rng(8)
    small = _c2_small(G, rng)
    large = [_problem("dual", 166, 20, M, 900 + M, rng) for M in (700, 1044)]
    assert np.all(_plan(G, "dual", 166, 20, [Y.shape[1] for Y, _ in small]) == 0)
    alone = [G.to_gpu_params(p) for _, p in small]
    G.vb.vbls_batched_([Y for Y, _ in small], alone, 20, full_cov=True, ctx=ctx)
    order = small[:10] + large[:1] + small[10:] + large[1:]
    mixed = [G.to_gpu_params(p) for _, p in order]
    G.vb.vbls_batched_([Y for Y, _ in order], mixed, 20, full_cov=True, ctx=ctx)
    got = mixed[:10] + mixed[11:-1]
    for a, b in zip(alone, got):
        sa, sb = _snap(a), _snap(b)
        for f in sa:
            assert np.array_equal(sa[f], sb[f]), f
    for (Y, p), q in zip(large, (mixed[10], mixed[-1])):
        vo.vbls(Y, p, 20, full_cov=True)
        G.compare(q, p, TOL, _fields("dual", False))


def test_large_batch_is_reproducible_and_independent_of_its_neighbours(G, ctx):
    rng = np.random.default_rng(9)
    large = [_problem("sparse", 166, 20, M, 40 + M, rng, diag_var=True) for M in (333, 1044)]
    others = _c2_small(G, rng, 6, "sparse", True)

    def run(items):
        qs = [G.to_gpu_params(p) for _, p in items]
        G.vb.vbls_batched_([Y for Y, _ in items], qs, 10, full_cov=True, diag_var=True, ctx=ctx)
        return qs

    r1, r2 = run(large), run(large)
    r3 = run(others[:3] + large[1:] + others[3:] + large[:1])
    for a, b in zip(r1, r2):
        sa, sb = _snap(a, "sparse"), _snap(b, "sparse")
        assert all(np.array_equal(sa[f], sb[f]) for f in sa)
    for a, b in ((r1[1], r3[3]), (r1[0], r3[-1])):
        sa, sb = _snap(a, "sparse"), _snap(b, "sparse")
        assert all(np.array_equal(sa[f], sb[f]) for f in sa)


def test_non_pd_in_a_large_bag(G, ctx):
    rng = np.random.default_rng(11)
    items = [_problem("sparse", 166, 20, M, 70 + M, rng) for M in (20, 700, 500)]
    items[1][1].CA[5] = -1e6                        # a negative prior precision: that column's precision is not PD
    qs = [G.to_gpu_params(p) for _, p in items]
    assert _plan(G, "sparse", 166, 20, [700])[0] > 0
    batch = G.vb.BatchedVbls([Y for Y, _ in items], qs, ctx=ctx, yhat=True)
    assert batch.run(3, full_cov=True) == -2
    batch.readback()
    assert np.isnan(np.asarray(qs[1].AHat)).any()
    for i in (0, 2):
        Y, p = items[i]
        vo.vbls(Y, p, 3, full_cov=True)
        G.compare(qs[i], p, TOL, _fields("sparse", False))


def test_arena_regrowth_large_small_large(G, ctx):
    rng = np.random.default_rng(12)
    batches = [[_problem("dual", 166, 20, M, 10 + M, rng) for M in (5, 800)],
               [_problem("dual", 166, 20, M, 20 + M, rng) for M in (3, 9)],
               [_problem("dual", 166, 20, M, 30 + M, rng) for M in (1044, 400, 12)]]
    for items in batches:
        qs = [G.to_gpu_params(p) for _, p in items]
        b = G.vb.BatchedVbls([Y for Y, _ in items], qs, ctx=ctx, yhat=True, keep_blocks=True)
        b.run(4, full_cov=True)
        b.readback()
        for (Y, p), q in zip(items, qs):
            vo.vbls(Y, p, 4, full_cov=True)
            G.compare(q, p, TOL, _fields("dual", False))
            assert G.rel(q.SigmaATVec_blocks, p.SigmaATVec_blocks) < TOL


def _oracle_copy_dual(Y, old):
    p = vo.vbmf_dual_init(Y, old.H, old.H0, gamma0=old.gamma0, delta0=old.delta0, eta0=old.eta0, zeta0=old.zeta0,
                          rng=np.random.default_rng(0))
    p.BHat, p.SigmaB, p.CB, p.gamma, p.delta = old.BHat.copy(), old.SigmaB.copy(), old.CB.copy(), old.gamma, old.delta.copy()
    p.alpha00, p.beta00, p.alpha01, p.beta01 = old.alpha00, old.beta00, old.alpha01, old.beta01
    return p


def test_classify_bags_musk2_shaped(G, ctx):
    """mil.classify_bags on Musk2-shaped bags (166 features, bags of 1..1044 instances), against the reference procedure
    spelled out with the oracle bag by bag, on a subset that includes the largest bag."""
    rng = np.random.default_rng(2)
    L, H, H0 = 166, 20, 19
    models = []
    for c in range(2):
        Yt = 10.0 * synth(L, 300, 3, seed=800 + c)
        p = vo.vbmf_dual_init(Yt, H, H0, rng=rng)
        vo.vbmf_dual_run(Yt, p, 8, eps=0.0, full_cov=True)
        models.append(p)
    gm = [G.to_gpu_params(m) for m in models]
    sizes = [1044, 2, 17, 350, 40, 640, 5, 90]
    bags = [np.asfortranarray(10.0 * synth(L, M, 3, seed=(800 if b % 2 == 0 else 801) + 7 * b)) for b, M in enumerate(sizes)]
    labels, e0, e1 = G.vb.mil.classify_bags(gm[0], gm[1], bags, class_alg="dual", ctx=ctx)
    for b in (0, 1, 3, 5):
        Y = bags[b]
        errs = []
        for m in models:
            p = _oracle_copy_dual(Y, m)
            vo.vbls(Y, p, 20, full_cov=True)
            errs.append(np.linalg.norm(p.YHat - Y, 2) / (Y.shape[0] * Y.shape[1]))
        assert abs(e0[b] - errs[0]) <= 1e-9 * errs[0] and abs(e1[b] - errs[1]) <= 1e-9 * errs[1]
        assert labels[b] == (0 if errs[0] < errs[1] else 1)
