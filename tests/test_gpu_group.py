"""Several solvers of one context run in lockstep (vbmf_b200_solver_run_group / run_group / vbmf_group_): one INT8 K1 and
one K2 per iteration serve every member.  A member's result depends only on its own state, Y and the group's total width, so
a group of one is bit for bit a solo run, and reordering or replacing the other members changes nothing in it."""
import copy
import os

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


def _fields(q):
    return {k: v for k, v in vars(q).items() if isinstance(v, (np.ndarray, float, int)) and k not in ("iterations", "d")}


def _same(a, b):
    fa, fb = _fields(a), _fields(b)
    assert fa.keys() == fb.keys()
    for k in fa:
        assert np.array_equal(np.asarray(fa[k]), np.asarray(fb[k]), equal_nan=True), k


def _solo(G, ctx, p, flags, niter, eps):
    q = copy.deepcopy(p)
    s = G.vb.Solver(ctx, q)
    try:
        s.upload(q)
        it, d = s.run(niter, eps, flags)
        s.download(q)
    finally:
        s.close()
    return q, it, d


def _group(G, ctx, ps, flags, niter, eps):
    qs = [copy.deepcopy(p) for p in ps]
    ss = [G.vb.Solver(ctx, q) for q in qs]
    try:
        for s, q in zip(ss, qs):
            s.upload(q)
        res = G.vb.run_group(ss, niter, eps, flags)
        for s, q in zip(ss, qs):
            s.download(q)
        failed = [s.failed for s in ss]
    finally:
        for s in ss:
            s.close()
    return qs, res, failed


def _flags(G, **kw):
    return G.vb.api._flags(**kw)


# kind, H0 (dual / trial), flag keywords: the flag sets of the teacher-forced tests
KINDS = [("dense", 0, dict(est_covs=True, est_var=True)), ("dense", 0, dict(est_var=True)), ("dense", 0, dict(est_covs=True)),
         ("sparse", 0, dict(est_cb=True)), ("sparse", 0, dict(full_cov=True, est_cb=True)), ("sparse", 0, dict()),
         ("sparse", 0, dict(full_cov=True, diag_var=True, est_cb=True)), ("sparse", 0, dict(diag_var=True, est_cb=True)),
         ("dual", 3, dict(est_priors=True, est_cb=True)), ("dual", 3, dict(full_cov=True, est_priors=True, est_cb=True)),
         ("dual", 3, dict(est_priors=True)), ("dual", 3, dict(diag_var=True, est_cb=True)),
         ("dual", 3, dict(full_cov=True, diag_var=True, est_priors=True, est_cb=True)),
         ("trial", 3, dict(est_priors=True)), ("trial", 3, dict(full_cov=True, est_priors=True)),
         ("trial", 3, dict(full_cov=True, diag_var=True, est_priors=True))]


def _init(G, kind, Y, H, H0, seed):
    rng = np.random.default_rng(seed)
    if kind == "dense":
        return G.vb.vbmf_init(Y, H, rng=rng)
    if kind == "sparse":
        return G.vb.vbmf_sparse_init(Y, H, rng=rng)
    if kind == "dual":
        return G.vb.vbmf_dual_init(Y, H, H0, rng=rng)
    return G.vb.vbmf_trial_init(Y, H, H0, Y.shape[1] // 3, rng=rng)


@pytest.mark.parametrize("H", [7, 64])
@pytest.mark.parametrize("kind,H0,kw", KINDS)
def test_group_of_one_is_solo(G, ctx, kind, H0, kw, H):
    Y = np.asfortranarray(synth(300, 1000, 4, seed=H))
    ctx.attach(Y, force=True)
    p = _init(G, kind, Y, H, H0, seed=3)
    f = _flags(G, **kw)
    qs, it_s, d_s = _solo(G, ctx, p, f, 8, 1e-12)
    (qg,), [(it_g, d_g)], failed = _group(G, ctx, [p], [f], 8, 1e-12)
    assert (it_g, d_g) == (it_s, d_s) and failed == [False]
    _same(qg, qs)


def test_group_of_one_is_solo_large(G, ctx):
    """3000 x 50000: the persistent CTAs walk several work items and split-K slabs."""
    ctx.synth(3000, 50000, rank=6, noise=0.1, seed=5)
    Y = ctx.download_Y()
    for kind, H0, kw in (KINDS[0], KINDS[4], KINDS[8]):
        p = _init(G, kind, Y, 24, H0, seed=4)
        f = _flags(G, **kw)
        qs, it_s, d_s = _solo(G, ctx, p, f, 3, 0.0)
        (qg,), [(it_g, d_g)], _ = _group(G, ctx, [p], [f], 3, 0.0)
        assert (it_g, d_g) == (it_s, d_s)
        _same(qg, qs)


def test_mixed_group_teacher_forced(G, ctx):
    """Dense H = 16, labelled sparse full_cov H = 8, dual H = 12 / H0 = 4 and trial H = 10 / H0 = 3 (total 46) in one group:
    from the oracle's state of every iteration, one group iteration matches the oracle's single iteration per member."""
    L, M = 60, 400
    Y = synth(L, M, 4, seed=21)
    Yf = np.asfortranarray(Y)
    ctx.attach(Yf, force=True)
    ps = [vo.vbmf_init(Y, 16, rng=np.random.default_rng(1)),
          vo.vbmf_sparse_init(Y, 8, H1=2, labels=list(range(2, M + 1, 4)), rng=np.random.default_rng(2)),
          vo.vbmf_dual_init(Y, 12, 4, rng=np.random.default_rng(3)),
          vo.vbmf_trial_init(Y, 10, 3, 150, rng=np.random.default_rng(4))]
    runs = [lambda s: vo.vbmf_run(Y, s, 1, eps=0.0, est_covs=True, est_var=True)[2],
            lambda s: vo.vbmf_sparse_run(Y, s, 1, eps=0.0, full_cov=True, est_cb=True)[0],
            lambda s: vo.vbmf_dual_run(Y, s, 1, eps=0.0, est_priors=True, est_cb=True)[0],
            lambda s: vo.vbmf_trial_run(Y, s, 1, eps=0.0, est_priors=True)[0]]
    flags = [_flags(G, est_covs=True, est_var=True), _flags(G, full_cov=True, est_cb=True),
             _flags(G, est_priors=True, est_cb=True), _flags(G, est_priors=True, est_cb=True)]
    for _ in range(10):
        qs = [G.to_gpu_params(p) for p in ps]
        d_o = [run(p) for run, p in zip(runs, ps)]
        qs, res, _ = _group(G, ctx, qs, flags, 1, 0.0)
        for q, p, (it, d), do in zip(qs, ps, res, d_o):
            assert it == 1
            G.compare(q, p, TOL)
            assert abs(d - do) <= 1e-9 + 1e-8 * abs(do)


def test_free_running_restarts(G, ctx):
    """Four dense H = 16 restarts: each stops at the oracle's iteration, and they stop at different iterations."""
    Y = synth(40, 200, 3, seed=77)
    ctx.attach(np.asfortranarray(Y), force=True)
    ps = [vo.vbmf_init(Y, 16, rng=np.random.default_rng(100 + s)) for s in range(4)]
    qs, res, _ = _group(G, ctx, [G.to_gpu_params(p) for p in ps], [0] * 4, 400, 1e-6)
    its = []
    for p, q, (it, d) in zip(ps, qs, res):
        po = copy.deepcopy(p)
        _, it_o, d_o = vo.vbmf_run(Y, po, 400, eps=1e-6)
        assert it == it_o
        its.append(it)
        floor = G.sensitivity(lambda s: vo.vbmf_run(Y, s, 400, eps=1e-6), p, ["AHat", "BHat"])
        G.compare(q, po, max(TOL, 100 * floor))
    assert len(set(its)) >= 2


def _isolation_case(G):
    Y = np.asfortranarray(synth(200, 3000, 4, seed=8))
    ps = [G.vb.vbmf_init(Y, 16, rng=np.random.default_rng(10)),
          G.vb.vbmf_sparse_init(Y, 8, rng=np.random.default_rng(11)),
          G.vb.vbmf_dual_init(Y, 12, 4, rng=np.random.default_rng(12)),
          G.vb.vbmf_init(Y, 16, rng=np.random.default_rng(13))]
    flags = [_flags(G, est_covs=True, est_var=True), _flags(G, diag_var=True, est_cb=True),
             _flags(G, full_cov=True, est_priors=True, est_cb=True), _flags(G, est_var=True)]
    return Y, ps, flags


def test_isolation_bit_for_bit(G, ctx):
    Y, ps, flags = _isolation_case(G)
    ctx.attach(Y, force=True)
    base, res, _ = _group(G, ctx, ps, flags, 6, 1e-12)
    # permuted
    perm = [2, 0, 3, 1]
    qp, resp, _ = _group(G, ctx, [ps[i] for i in perm], [flags[i] for i in perm], 6, 1e-12)
    for j, i in enumerate(perm):
        _same(qp[j], base[i])
        assert resp[j] == res[i]
    # another state of the same H in slot 3
    other = G.vb.vbmf_init(Y, 16, rng=np.random.default_rng(99))
    qo, reso, _ = _group(G, ctx, ps[:3] + [other], flags, 6, 1e-12)
    for i in range(3):
        _same(qo[i], base[i])
        assert reso[i] == res[i]
    # a member whose first precision is not positive definite: -2, NaN in that member only
    bad = G.vb.vbmf_init(Y, 16, rng=np.random.default_rng(98))
    bad.invCA = np.asfortranarray(-1e6 * np.eye(16))
    with pytest.warns(G.vb.VBMFWarning):
        qb, resb, failed = _group(G, ctx, ps[:3] + [bad], flags, 6, 1e-12)
    assert failed == [False, False, False, True]
    assert np.isnan(qb[3].SigmaA).any()
    for i in range(3):
        _same(qb[i], base[i])
        assert resb[i] == res[i]


def test_dmma_path_matches_solo(G, monkeypatch):
    monkeypatch.setenv("VBMF_B200_GEMM", "dmma")
    c = G.vb.Context(device=0)
    monkeypatch.delenv("VBMF_B200_GEMM")
    try:
        Y, ps, flags = _isolation_case(G)
        c.attach(Y, force=True)
        qs, res, _ = _group(G, c, ps, flags, 5, 1e-12)
        for p, f, q, r in zip(ps, flags, qs, res):
            q1, it, d = _solo(G, c, p, f, 5, 1e-12)
            _same(q, q1)
            assert r == (it, d)
    finally:
        c.close()


def test_refusals_leave_state(G, ctx):
    Y = np.asfortranarray(synth(50, 300, 3, seed=2))
    ctx.attach(Y, force=True)
    p40, p32 = G.vb.vbmf_init(Y, 40, rng=np.random.default_rng(1)), G.vb.vbmf_sparse_init(Y, 32, rng=np.random.default_rng(2))
    s40, s32 = G.vb.Solver(ctx, p40), G.vb.Solver(ctx, p32)
    c2 = G.vb.Context(device=0)
    try:
        s40.upload(p40)
        s32.upload(p32)
        with pytest.raises(G.vb.VBMFError, match="add up to 72"):
            G.vb.run_group([s40, s32], 5)
        with pytest.raises(G.vb.VBMFError, match="appears twice"):
            G.vb.run_group([s40, s40], 5)
        with pytest.raises(G.vb.VBMFError, match="n >= 1"):
            G.vb.run_group([], 5)
        c2.attach(Y, force=True)
        p8 = G.vb.vbmf_init(Y, 8, rng=np.random.default_rng(3))
        s8 = G.vb.Solver(c2, p8)
        s8.upload(p8)
        with pytest.raises(G.vb.VBMFError, match="one context"):
            G.vb.run_group([s40, s8], 5)
        s8.close()
        for s, p in ((s40, p40), (s32, p32)):
            q = copy.deepcopy(p)
            s.download(q)
            _same(q, p)
        c2.set_shape(50, 300)
        s8 = G.vb.Solver(c2, p8)
        s8.upload(p8)
        with pytest.raises(G.vb.VBMFError, match="no Y attached"):
            G.vb.run_group([s8], 5)
        q = copy.deepcopy(p8)
        s8.download(q)
        _same(q, p8)
        s8.close()
    finally:
        s40.close()
        s32.close()
        c2.close()


def test_vbmf_group_yhat_and_options(G, ctx):
    Y = np.asfortranarray(synth(80, 500, 3, seed=5))
    ps = [G.vb.vbmf_init(Y, 8, rng=np.random.default_rng(1)), G.vb.vbmf_sparse_init(Y, 6, rng=np.random.default_rng(2))]
    solo = [copy.deepcopy(p) for p in ps]
    G.vb.vbmf_group_(Y, ps, 7, eps=1e-12, options=[dict(est_covs=True), dict(full_cov=True)], ctx=ctx, yhat=True)
    G.vb.vbmf_(Y, solo[0], 7, eps=1e-12, est_covs=True, ctx=ctx)
    G.vb.vbmf_sparse_(Y, solo[1], 7, eps=1e-12, full_cov=True, ctx=ctx)
    for p, s in zip(ps, solo):
        assert p.iterations == 7 and p.failed is False
        assert G.rel(p.YHat, p.BHat @ p.AHat.T) < 1e-13
        for f in ("AHat", "BHat", "SigmaA", "SigmaB", "YHat"):
            assert np.array_equal(getattr(p, f), getattr(s, f)), f
    with pytest.raises(TypeError):
        G.vb.vbmf_group_(Y, ps[:1], 1, options=[dict(diag_var=True)], ctx=ctx)


def test_repeated_groups_do_not_grow_memory(G, ctx):
    import torch
    Y = np.asfortranarray(synth(500, 4000, 3, seed=6))
    ctx.attach(Y, force=True)
    ps = [G.vb.vbmf_init(Y, 16, rng=np.random.default_rng(s)) for s in range(4)]

    def cycle():
        _group(G, ctx, ps, [0] * 4, 3, 0.0)
    cycle()
    ctx.sync()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(40):
        cycle()
    ctx.sync()
    assert free0 - torch.cuda.mem_get_info(0)[0] <= 32 << 20
