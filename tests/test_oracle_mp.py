"""The NumPy oracle against a second, independent 40-digit restatement (oracle/mp_restatement.py) on the branches the
reference's own golden logs do not exercise (SURVEY section 8(c): "parity unpinned" branches)."""
import copy

import numpy as np
import pytest

from oracle import vbmf_oracle as vo
from oracle import mp_restatement as mr

TOL = 1e-12


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _cmp(p, d, fields, tol=TOL):
    for f in fields:
        got = getattr(p, f)
        want = mr.to_float(d[f])
        assert _rel(np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)) <= tol, f


def _problem(L, M, H, seed):
    rng = np.random.default_rng(seed)
    Y = rng.standard_normal((L, 2)) @ rng.standard_normal((2, M)) + 0.1 * rng.standard_normal((L, M))
    return np.ascontiguousarray(Y), rng


SPARSE_FIELDS = ("AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "BHat", "SigmaB", "CA", "beta", "CB", "delta")


@pytest.mark.parametrize("full_cov", [False, True])
@pytest.mark.parametrize("diag_var", [False, True])
def test_sparse_steps_match_high_precision_restatement(full_cov, diag_var):
    L, M, H = 5, 4, 3
    Y, rng = _problem(L, M, H, 11)
    p = vo.vbmf_sparse_init(Y, H, H1=1, labels=[2, 4], rng=rng)
    p.sigmaVecHat = 0.5 + rng.random(L)          # a non-trivial heteroscedastic state
    p.CA = 0.5 + rng.random(M * H)
    for it in range(3):
        Ym, d = mr.from_oracle(copy.deepcopy(p), Y)   # teacher forcing: both start every iteration from the same state
        vo.sparse_updateA(Y, p, full_cov=full_cov, diag_var=diag_var)
        vo.sparse_updateB(Y, p, diag_var=diag_var)
        vo.sparse_updateCA(p)
        vo.sparse_updateCB(p)
        vo.sparse_updateSigma(Y, p, diag_var=diag_var)
        mr.updateA(Ym, d, full_cov=full_cov, diag_var=diag_var)
        mr.updateB(Ym, d, diag_var=diag_var)
        mr.updateCA(d)
        mr.updateCB(d)
        mr.updateSigma(Ym, d, diag_var=diag_var)
        _cmp(p, d, SPARSE_FIELDS)
        _cmp(p, d, ("sigmaVecHat", "zetaVec") if diag_var else ("sigmaHat", "zeta"))


def test_q2_repeat_inner_tail_is_not_a_tiling():
    """The literal `repeat(d[1:H], inner = M-1)` (src/vbmf_sparse.jl:221) and the oracle's index map agree, and differ
    from the tiling one would expect - the quirk is real and replicated."""
    L, M, H = 4, 5, 3
    Y, rng = _problem(L, M, H, 5)
    p = vo.vbmf_sparse_init(Y, H, rng=rng)
    p.SigmaB = np.diag(rng.random(H))
    Ym, d = mr.from_oracle(copy.deepcopy(p), Y)
    vo.sparse_updateA(Y, p, full_cov=False)
    mr.updateA(Ym, d, full_cov=False)
    _cmp(p, d, ("diagSigmaATVec", "ATVecHat", "SigmaA"))
    prec = 1.0 / p.diagSigmaATVec - 1.0           # CA == 1
    assert not np.allclose(prec, np.tile(prec[:H], M))


def test_sparse_lower_bound_literal_kron_determinant():
    L, M, H = 4, 3, 2
    Y, rng = _problem(L, M, H, 3)
    p = vo.vbmf_sparse_init(Y, H, rng=rng, alpha0=1e-3, beta0=1e-3, gamma0=1e-3, delta0=1e-3, eta0=1e-3, zeta0=1e-3)
    vo.vbmf_sparse_run(Y, p, 4, eps=0.0, full_cov=True)
    Ym, d = mr.from_oracle(p, Y)
    want = float(mr.lowerBound(Ym, d))
    got = vo.sparse_lowerBound(Y, p)
    assert abs(got - want) <= 1e-11 * abs(want)


def test_dual_grouped_ard_and_hyperprior_root():
    L, M, H, H0 = 5, 4, 3, 2
    Y, rng = _problem(L, M, H, 17)
    p = vo.vbmf_dual_init(Y, H, H0, rng=rng, alpha0=1.0, beta0=1.0)
    for it in range(3):
        Ym, d = mr.from_oracle(copy.deepcopy(p), Y)
        vo.dual_updateA(Y, p, full_cov=(it % 2 == 1))
        vo.sparse_updateB(Y, p)
        vo.dual_updateCA(p)
        vo.sparse_updateCB(p)
        vo.sparse_updateSigma(Y, p)
        vo.dual_updateAlpha00(p); vo.dual_updateAlpha01(p); vo.dual_updateBeta00(p); vo.dual_updateBeta01(p)
        mr.updateA(Ym, d, full_cov=(it % 2 == 1), mask=False)
        mr.updateB(Ym, d)
        mr.dual_updateCA(d)
        mr.updateCB(d)
        mr.updateSigma(Ym, d)
        mr.dual_update_priors(d)
        _cmp(p, d, SPARSE_FIELDS + ("CA0", "CA1", "beta0", "beta1", "alpha0", "alpha1", "sigmaHat"))
        _cmp(p, d, ("alpha00", "alpha01", "beta00", "beta01"), tol=1e-10)


@pytest.mark.parametrize("M0", [0, 2, 5])
def test_trial_three_group_ard_and_priors(M0):
    """src/vbmf_trial.jl: groups (columns < H0 | rows <= M0 | rows > M0) incl. the empty-group edges M0 = 0 and M0 = M."""
    L, M, H, H0 = 4, 5, 3, 1
    Y, rng = _problem(L, M, H, 23 + M0)
    p = vo.vbmf_trial_init(Y, H, H0, M0, rng=rng, alpha0=1.0, beta0=1.0)
    for it in range(3):
        Ym, d = mr.from_oracle(copy.deepcopy(p), Y)
        vo.trial_updateA(Y, p, full_cov=(it == 1))
        vo.sparse_updateB(Y, p)
        vo.trial_updateCA(p)
        vo.sparse_updateCB(p)
        vo.sparse_updateSigma(Y, p)
        vo.trial_update_priors(p)
        mr.updateA(Ym, d, full_cov=(it == 1), mask=False)
        mr.trial_split(d)
        mr.updateB(Ym, d)
        mr.trial_updateCA(d)
        mr.updateCB(d)
        mr.updateSigma(Ym, d)
        mr.trial_update_priors(d)
        _cmp(p, d, ("AHat", "diagSigmaATVec", "SigmaA", "BHat", "SigmaB", "CA", "beta", "CA1", "beta1", "alpha1", "alpha2", "alpha3", "sigmaHat"))
        for f in ("CA2", "beta2", "CA3", "beta3"):
            if len(d[f]):
                _cmp(p, d, (f,))
        live = ["alpha01", "beta01"] + (["alpha02", "beta02"] if M0 > 0 else []) + (["alpha03", "beta03"] if M0 < M else [])
        _cmp(p, d, live, tol=1e-10)


def test_dual_lower_bound_literal():
    L, M, H, H0 = 4, 3, 3, 2
    Y, rng = _problem(L, M, H, 31)
    p = vo.vbmf_dual_init(Y, H, H0, rng=rng, alpha0=1e-2, beta0=1e-2, gamma0=1e-2, delta0=1e-2, eta0=1e-2, zeta0=1e-2)
    vo.vbmf_dual_run(Y, p, 4, eps=0.0, full_cov=True)
    Ym, d = mr.from_oracle(p, Y)
    want = float(mr.dual_lowerBound(Ym, d))
    got = vo.dual_lowerBound(Y, p)
    assert abs(got - want) <= 1e-11 * abs(want)


GOLDEN_SHA256 = {   # content of tests/golden/*.npz as decoded from the reference's .jld logs (see the test below)
    "vbmf_test": "3989a1a74c27586734db202ad24e1ee19eb6a453893b0a9aadf2a79d1a404f4f",
    "sparse_test": "81db05bf56b4494d92085226d44d04c317b52b21463472b5e40f5683403dd5be",
}


def test_golden_fixtures_match_the_decoded_reference_logs():
    """Every golden comparison rests on tests/golden/*.npz holding exactly what make_golden.py decoded from the reference's .jld
    logs.  The .jld files are not part of this repository, so the decoded content is pinned by digest: any edit to a fixture
    (a field, dtype, shape or value) fails here on every machine."""
    import hashlib
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    for name, want in GOLDEN_SHA256.items():
        g = np.load(os.path.join(here, "golden", name + ".npz"))
        h = hashlib.sha256()
        for k in sorted(g.files):
            a = np.ascontiguousarray(g[k])
            h.update(("%s|%s|%s|" % (k, a.dtype.str, a.shape)).encode())
            h.update(a.tobytes())
        assert h.hexdigest() == want, name


def test_golden_fixtures_regenerate_from_the_reference(tmp_path):
    """tests/golden/*.npz are exactly what tests/golden/make_golden.py decodes from the reference's own .jld logs (skipped unless
    VBMF_REFERENCE_DIR names a checkout of VBMatrixFactorization.jl; the .jld files are not part of this repository)."""
    import os
    import subprocess
    import sys
    ref = os.environ.get("VBMF_REFERENCE_DIR", "")
    if not ref or not os.path.isdir(os.path.join(ref, "examples", "data")):
        pytest.skip("VBMF_REFERENCE_DIR does not name a checkout of VBMatrixFactorization.jl")
    here = os.path.dirname(os.path.abspath(__file__))
    script = os.path.join(here, "golden", "make_golden.py")
    r = subprocess.run([sys.executable, script, "--out", str(tmp_path)], capture_output=True, text=True, timeout=300)
    if r.returncode != 0 and "--out" in (r.stderr + r.stdout):
        pytest.skip("make_golden.py has no --out option")
    assert r.returncode == 0, r.stderr[-500:]
    for name in ("vbmf_test.npz", "sparse_test.npz"):
        a, b = np.load(os.path.join(here, "golden", name)), np.load(os.path.join(str(tmp_path), name))
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert np.array_equal(a[k], b[k]), (name, k)
