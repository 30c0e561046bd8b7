"""Batched vbls! on labelled dense / sparse problems (AHat[labels, H-H1+1:H] = 0 after every A update, src/vbmf.jl:101,
src/vbmf_sparse.jl:245) and on dense states whose invCA is not diagonal (the first updateA! reads the whole matrix,
src/vbmf.jl:96), against the oracle's vbls and against vbls_ run on each problem alone."""
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
    G.vb._lib.check(lib.vbmf_b200_batched_plan({"dense": 0, "sparse": 1}[kind], L, H, int(full_cov), int(diag_var), M.size,
                                               M.ctypes.data, out.ctypes.data))
    return out


def _labels(i, M, rng):
    """Problem i's labels: none, every column, the first / middle / last columns, or a random subset."""
    k = i % 4
    if k == 0:
        return []
    if k == 1:
        return list(range(1, M + 1))
    if k == 2:
        return sorted({1, (M + 1) // 2, M})
    return sorted(set(int(x) for x in rng.integers(1, M + 1, size=max(1, M // 3))))


def _problem(kind, L, H, M, seed, rng, H1=0, labels=(), diag_var=False):
    Y = 10.0 * synth(L, M, min(3, H), seed=seed)
    if kind == "sparse":
        p = vo.vbmf_sparse_init(Y, H, H1=H1, labels=labels, rng=rng)
        p.sigmaHat = 0.7
        if diag_var:
            p.sigmaVecHat = rng.uniform(0.5, 2.0, L)
    else:
        p = vo.vbmf_init(Y, H, sigma2=0.9, H1=H1, labels=labels, rng=rng)
    p.SigmaB = np.diag(rng.uniform(1e-3, 1e-2, H))
    return np.asfortranarray(Y), p


def _fields(kind, diag_var):
    if kind == "dense":
        return ["AHat", "SigmaA", "CA", "invCA", "sigma2"]
    f = ["AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "CA", "beta", "sigmaHat", "zeta"]
    return f + (["sigmaVecHat", "zetaVec"] if diag_var else [])


def _snap(q, fields):
    return {f: np.array(getattr(q, f), dtype=np.float64, copy=True) for f in fields}


def _run(G, ctx, Ys, ps, niter, full_cov, diag_var):
    qs = [G.to_gpu_params(p) for p in ps]
    G.vb.vbls_batched_(list(Ys), qs, niter, full_cov=full_cov, diag_var=diag_var, ctx=ctx, yhat=True,
                       keep_blocks=full_cov and ps[0].kind == "sparse")
    return qs


LABEL_CASES = [  # kind, full_cov, diag_var, L, H, Ms: every case mixes one-CTA problems and cluster problems
    ("sparse", True, False, 166, 20, [1, 7, 300, 700, 1044]),
    ("sparse", False, True, 166, 21, [7, 300, 1044, 40]),
    ("sparse", True, True, 166, 13, [2, 40, 700, 9]),
    ("sparse", False, False, 38, 64, [2, 40, 200, 1]),
    ("sparse", True, False, 38, 64, [2, 40, 200, 3]),
    ("sparse", False, False, 166, 1, [3, 50, 9000, 4]),
    ("dense", False, False, 166, 20, [1, 7, 300, 700, 1044]),
    ("dense", False, False, 166, 32, [7, 267, 600, 30]),
    ("dense", False, False, 166, 7, [3, 40, 2000, 11]),
    ("dense", False, False, 166, 1, [5, 13000, 2, 9]),
]


@pytest.mark.parametrize("h1", ["one", "all"])
@pytest.mark.parametrize("kind,full_cov,diag_var,L,H,Ms", LABEL_CASES)
def test_labels_match_oracle_and_single_solver(G, ctx, kind, full_cov, diag_var, L, H, Ms, h1):
    H1 = 1 if h1 == "one" else H
    niter = 8
    cs = _plan(G, kind, L, H, Ms, full_cov, diag_var)
    assert np.any(cs == 0) and np.any(cs > 0), cs
    rng = np.random.default_rng(L + H + len(Ms) + H1)
    items = [_problem(kind, L, H, M, 500 + i, rng, H1, _labels(i, M, rng), diag_var) for i, M in enumerate(Ms)]
    Ys = [Y for Y, _ in items]
    ps = [p for _, p in items]
    assert any(p.labels.size == 0 for p in ps) and any(p.labels.size == p.M for p in ps)
    fields = _fields(kind, diag_var)
    qs = _run(G, ctx, Ys, ps, niter, full_cov, diag_var)

    # the unlabelled problems compute bit for bit what they compute in a call without any labels
    bare = []
    for p in ps:
        b = G.to_gpu_params(p)
        b.labels = np.zeros(0, dtype=np.int64)
        bare.append(b)
    G.vb.vbls_batched_(Ys, bare, niter, full_cov=full_cov, diag_var=diag_var, ctx=ctx, yhat=True)
    for p, q, b in zip(ps, qs, bare):
        if p.labels.size == 0:
            sq, sb = _snap(q, fields + ["YHat"]), _snap(b, fields + ["YHat"])
            assert all(np.array_equal(sq[f], sb[f]) for f in sq)

    for Y, p, q in zip(Ys, ps, qs):
        single = G.to_gpu_params(p)
        G.vb.vbls_(Y, single, niter, full_cov=full_cov, diag_var=diag_var, ctx=ctx)
        vo.vbls(Y, p, niter, full_cov=full_cov, diag_var=diag_var)
        if p.labels.size:
            assert np.all(np.asarray(q.AHat)[p.labels - 1, H - H1:] == 0.0)
        G.compare(q, p, TOL, fields)
        assert G.rel(q.YHat, p.YHat) < TOL
        if full_cov and kind == "sparse":
            assert G.rel(q.SigmaATVec_blocks, p.SigmaATVec_blocks) < TOL
        errs = {f: G.rel(getattr(q, f), getattr(single, f)) for f in fields + ["YHat"]}
        assert all(e <= 2 * TOL for e in errs.values()), errs


def _spd(rng, H):
    Q = rng.standard_normal((H, H))
    return np.asfortranarray(Q @ Q.T / H + 0.5 * np.eye(H))


@pytest.mark.parametrize("niter", [0, 1, 20])
@pytest.mark.parametrize("H", [7, 32])
def test_full_invCA_matches_oracle(G, ctx, H, niter):
    L, Ms = 166, [5, 40, 2000, 1044, 13]
    cs = _plan(G, "dense", L, H, Ms)
    assert np.any(cs == 0) and np.any(cs > 0), cs
    rng = np.random.default_rng(40 + H + niter)
    items = []
    for i, M in enumerate(Ms):
        labels = _labels(2, M, rng) if i == 3 else []
        Y, p = _problem("dense", L, H, M, 900 + i, rng, H1=2 if labels else 0, labels=labels)
        if i % 2 == 0:
            p.invCA = _spd(rng, H)        # CA stays diagonal, as updateCA! keeps it
        items.append((Y, p))
    Ys = [Y for Y, _ in items]
    ps = [p for _, p in items]
    before = [_snap(G.to_gpu_params(p), _fields("dense", False) + ["AHat"]) for p in ps]
    qs = _run(G, ctx, Ys, ps, niter, False, False)
    for Y, p, q, b in zip(Ys, ps, qs, before):
        if niter == 0:
            s = _snap(q, list(b))
            assert all(np.array_equal(s[f], b[f]) for f in b)
            continue
        vo.vbls(Y, p, niter)
        G.compare(q, p, TOL, _fields("dense", False))
        assert G.rel(q.YHat, p.YHat) < TOL
        ic = np.asarray(q.invCA)
        assert np.all(ic[~np.eye(H, dtype=bool)] == 0.0)


@pytest.mark.parametrize("H", [7, 32])
def test_diagonal_invCA_problem_does_not_depend_on_its_batch(G, ctx, H):
    """A problem with a diagonal invCA computes the same bits whether or not the call also holds full-invCA problems."""
    rng = np.random.default_rng(60 + H)
    items = [_problem("dense", 166, H, M, 950 + i, rng) for i, M in enumerate((6, 2000, 30))]
    alone = _run(G, ctx, [items[0][0], items[2][0]], [items[0][1], items[2][1]], 5, False, False)
    items[1][1].invCA = _spd(rng, H)
    mixed = _run(G, ctx, [Y for Y, _ in items], [p for _, p in items], 5, False, False)
    fields = _fields("dense", False) + ["YHat"]
    for a, b in zip(alone, (mixed[0], mixed[2])):
        sa, sb = _snap(a, fields), _snap(b, fields)
        assert all(np.array_equal(sa[f], sb[f]) for f in sa)


def test_states_refused_as_solver_creation_refuses_them(G, ctx):
    rng = np.random.default_rng(8)
    for kind in ("sparse", "dense"):
        items = [_problem(kind, 38, 6, M, 75 + i, rng) for i, M in enumerate((12, 40))]
        items[1][1].labels = np.array([41], dtype=np.int64)          # checked even with H1 = 0, as vbls_ checks it
        with pytest.raises(G.vb.VBMFError, match=r"label 41 of problem 1 out of range 1\.\.40"):
            G.vb.vbls_batched_([Y for Y, _ in items], [G.to_gpu_params(p) for _, p in items], 3, ctx=ctx)
        items[1][1].labels = np.array([2], dtype=np.int64)
        for h1 in (7, -1):
            items[1][1].H1 = h1
            with pytest.raises(G.vb.VBMFError, match=r"H1 of problem 1 must be in 0\.\.H"):
                G.vb.vbls_batched_([Y for Y, _ in items], [G.to_gpu_params(p) for _, p in items], 3, ctx=ctx)
    # a dense CA with off-diagonal entries: updateCA! would invert all of it, the batched kernels keep CA diagonal
    items = [_problem("dense", 38, 6, M, 77 + i, rng) for i, M in enumerate((12, 40))]
    items[0][1].CA[1, 2] = items[0][1].CA[2, 1] = 0.1
    with pytest.raises(G.vb.VBMFError, match=r"CA of problem 0 is not diagonal"):
        G.vb.vbls_batched_([Y for Y, _ in items], [G.to_gpu_params(p) for _, p in items], 3, ctx=ctx)


def test_out_of_range_label_names_the_problem(G, ctx):
    rng = np.random.default_rng(5)
    for kind in ("sparse", "dense"):
        for bad in (0, -3, 41):
            items = [_problem(kind, 38, 6, M, 70 + i, rng, 2, [1, M]) for i, M in enumerate((12, 40, 40))]
            items[2][1].labels = np.array([3, bad], dtype=np.int64)
            qs = [G.to_gpu_params(p) for _, p in items]
            with pytest.raises(G.vb.VBMFError, match=r"label %d of problem 2 out of range 1\.\.40" % bad):
                G.vb.vbls_batched_([Y for Y, _ in items], qs, 3, ctx=ctx)


def test_non_pd_full_invCA_fails_its_problem_only(G, ctx):
    rng = np.random.default_rng(6)
    H = 9
    items = [_problem("dense", 166, H, M, 80 + i, rng) for i, M in enumerate((20, 2000, 30, 1044))]
    for j in (1, 2):                          # indefinite: unit diagonal, off-diagonal entries of 1e6
        ic = np.eye(H)
        ic[0, 1] = ic[1, 0] = 1e6
        items[j][1].invCA = np.asfortranarray(ic)
    items[3][1].invCA = _spd(rng, H)
    qs = [G.to_gpu_params(p) for _, p in items]
    batch = G.vb.BatchedVbls([Y for Y, _ in items], qs, ctx=ctx, yhat=True)
    assert batch.run(4) == -2
    batch.readback()
    for j in (1, 2):
        assert np.isnan(np.asarray(qs[j].AHat)).all() and np.isnan(np.asarray(qs[j].SigmaA)).all()
    for j in (0, 3):
        Y, p = items[j]
        vo.vbls(Y, p, 4)
        G.compare(qs[j], p, TOL, _fields("dense", False))


@pytest.mark.parametrize("kind", ["dual", "trial"])
def test_dual_and_trial_ignore_labels(G, ctx, kind):
    """Dual and trial states have no labels (their C structs carry none): labels set on the Python parameter objects stay
    out of the call, so the results are those of the same states without them."""
    rng = np.random.default_rng(7)
    items = []
    for i, M in enumerate((9, 30, 700)):
        Y = np.asfortranarray(10.0 * synth(166, M, 3, seed=60 + i))
        p = vo.vbmf_dual_init(Y, 12, 11, rng=rng) if kind == "dual" else vo.vbmf_trial_init(Y, 12, 10, M // 2, rng=rng)
        p.SigmaB = np.diag(rng.uniform(1e-3, 1e-2, 12))
        p.sigmaHat = 0.7
        items.append((Y, p))
    plain = [G.to_gpu_params(p) for _, p in items]
    labelled = [G.to_gpu_params(p) for _, p in items]
    for q in labelled:
        q.labels = np.arange(1, q.M + 1, dtype=np.int64)
    for qs in (plain, labelled):
        G.vb.vbls_batched_([Y for Y, _ in items], qs, 6, full_cov=True, ctx=ctx)
    fields = ["AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "CA", "beta", "sigmaHat", "zeta", "YHat"]
    for a, b in zip(plain, labelled):
        sa, sb = _snap(a, fields), _snap(b, fields)
        assert all(np.array_equal(sa[f], sb[f]) for f in sa)
