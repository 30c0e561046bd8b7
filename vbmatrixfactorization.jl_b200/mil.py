"""The callers of the hot path in the reference's MIL example (examples/mil_util.jl), on top of the B200 library.

SURVEY section 8(f) N1: `vbls!` (:179-203), `copy_vbmf_params` (:212-293), `train_dual` with its restarts (:327-385) and the
classification loop built from them (`classify` :453-535, `test_classification` :557-588).  The reference classifies one bag
at a time - two `vbls!` calls per bag, each a handful of tiny matrix products; here `classify_bags` puts every (bag, class
model) pair of a whole test set into ONE call of `vbmf_b200_batched_vbls`: one launch of the one-CTA-per-problem kernel, plus
the wide kernel (one thread-block cluster per bag) for bags too large for one CTA's shared memory.

Only the VB-based classifiers are mirrored ("vbls", "dual"); "ols"/"rls" are two-line host least-squares formulas with no VB
update in them and stay with the caller.  The matrix norms of the L x M residuals follow Julia 0.5 (`norm(::Matrix)` =
spectral norm, SURVEY quirk Q1) and are evaluated here on the host, one LAPACK SVD per bag and class model.  That is not
cheap: on the Musk2-shaped batch of tools/batched/large_bags.py it takes about 1 s per pair of class models, against
15 ms for `residual_norm_batched` / `BatchedVbls.residual_norm`, which compute the same norms on the device without
downloading YHat (DESIGN section 5).
"""
import numpy as np

from . import _lib as L_
from . import api as A


def _cp(x):
    return np.array(x, dtype=np.float64, order="F", copy=True)


def copy_vbmf_params(Y, old_params, rng=None):
    """`copy_vbmf_params(Y, old_params)` examples/mil_util.jl:212-293: a fresh parameter object for the bag Y (its own M) that
    carries the trained basis (BHat, SigmaB, CB, ...) and hyper-priors of `old_params`.  Trial parameters give a PAIR
    (params0 with the priors of group 2, params1 with group 3's priors in group 2's place), as in the reference."""
    Y = np.asarray(Y)
    k = old_params.kind
    if k == L_.DENSE:
        # labels and H1 are deliberately not copied (:214-215)
        p = A.vbmf_init(Y, old_params.H, sigma2=old_params.sigma2, rng=rng)
        p.BHat, p.SigmaB = _cp(old_params.BHat), _cp(old_params.SigmaB)
        p.CB, p.invCB = _cp(old_params.CB), _cp(old_params.invCB)
        return p
    if k == L_.SPARSE:
        p = A.vbmf_sparse_init(Y, old_params.H, alpha0=old_params.alpha0, beta0=old_params.beta0, gamma0=old_params.gamma0,
                               delta0=old_params.delta0, eta0=old_params.eta0, zeta0=old_params.zeta0, rng=rng)
        p.BHat, p.SigmaB = _cp(old_params.BHat), _cp(old_params.SigmaB)
        p.CB, p.gamma, p.delta = np.array(old_params.CB, dtype=np.float64), old_params.gamma, np.array(old_params.delta, dtype=np.float64)
        return p            # (`params.invCB = ...` at :232 names a field sparse parameters do not have: quirk Q10, ignored)
    if k == L_.DUAL:
        p = A.vbmf_dual_init(Y, old_params.H, old_params.H0, gamma0=old_params.gamma0, delta0=old_params.delta0,
                             eta0=old_params.eta0, zeta0=old_params.zeta0, rng=rng)
        p.BHat, p.SigmaB = _cp(old_params.BHat), _cp(old_params.SigmaB)
        p.CB, p.gamma, p.delta = np.array(old_params.CB, dtype=np.float64), old_params.gamma, np.array(old_params.delta, dtype=np.float64)
        p.alpha00, p.beta00, p.alpha01, p.beta01 = old_params.alpha00, old_params.beta00, old_params.alpha01, old_params.beta01
        return p
    if k == L_.TRIAL:
        M = Y.shape[1]
        out = []
        for which in (0, 1):
            p = A.vbmf_trial_init(Y, old_params.H, old_params.H0, M, gamma0=old_params.gamma0, delta0=old_params.delta0,
                                  eta0=old_params.eta0, zeta0=old_params.zeta0, rng=rng)
            p.BHat, p.SigmaB = _cp(old_params.BHat), _cp(old_params.SigmaB)
            p.CB, p.gamma, p.delta = np.array(old_params.CB, dtype=np.float64), old_params.gamma, np.array(old_params.delta, dtype=np.float64)
            p.alpha01, p.beta01 = old_params.alpha01, old_params.beta01
            if which == 0:
                p.alpha02, p.beta02 = old_params.alpha02, old_params.beta02
            else:
                p.alpha02, p.beta02 = old_params.alpha03, old_params.beta03
            p.alpha03, p.beta03 = 1e-10, 1e-10
            out.append(p)
        return tuple(out)
    raise L_.VBMFError("copy_vbmf_params: unknown parameter type")


def _spectral(X):
    X = np.asarray(X, dtype=np.float64)
    return float(np.linalg.norm(X, 2)) if X.size else 0.0


def classify_bags(res0, res1, Ys, class_alg="dual", ctx=None, rng=None):
    """`classify(res0, res1, Y; class_alg)` (examples/mil_util.jl:453-535) for a whole list of bags in two batched launches
    (one per class model).  class_alg = "dual": `vbls!(Y, params, 20, full_cov = true)` on copies of both models, label 0
    iff ||YHat0 - Y||/(L*M) < ||YHat1 - Y||/(L*M) (:519-533).  class_alg = "vbls": 150 iterations, label 1 iff
    ||Y - B0*A0'|| > ||Y - B1*A1'|| (:470-492).  Returns (labels, err0, err1) as arrays."""
    if class_alg not in ("dual", "vbls"):
        raise L_.VBMFError('classify: only the VB classifiers "dual" and "vbls" run on the device')
    Ys = [np.asfortranarray(np.asarray(Y, dtype=np.float64)) for Y in Ys]
    niter, full_cov = (20, True) if class_alg == "dual" else (150, False)
    errs = []
    for res in (res0, res1):
        if res.kind == L_.TRIAL:
            raise L_.VBMFError("classify: trial parameters are classified through factorize/vbls_ directly (copy_vbmf_params gives a pair)")
        ps = [copy_vbmf_params(Y, res, rng=rng) for Y in Ys]
        A.vbls_batched_(Ys, ps, niter, full_cov=full_cov, ctx=ctx, yhat=True)
        if class_alg == "dual":
            errs.append(np.array([_spectral(p.YHat - Y) / (Y.shape[0] * Y.shape[1]) for p, Y in zip(ps, Ys)]))
        else:
            errs.append(np.array([_spectral(Y - np.asarray(res.BHat) @ np.asarray(p.AHat).T) for p, Y in zip(ps, Ys)]))
    err0, err1 = errs
    if class_alg == "dual":
        labels = np.where(err0 < err1, 0, 1)
    else:
        labels = np.where(err0 > err1, 1, 0)
    return labels.astype(np.int64), err0, err1


def classify(res0, res1, Y, threshold=1e-1, class_alg="dual", ctx=None, rng=None):
    """Single-bag form with the reference's signature and return value `(label, err0, err1)`."""
    labels, e0, e1 = classify_bags(res0, res1, [Y], class_alg=class_alg, ctx=ctx, rng=rng)
    return int(labels[0]), float(e0[0]), float(e1[0])


def test_classification(res0, res1, Ys, labels, class_alg="dual", ctx=None, rng=None):
    """`test_classification` examples/mil_util.jl:557-588 on explicit bags: (mer, eer, fp, fn, n0, n1)."""
    labels = np.asarray(labels, dtype=np.int64)
    est, _, _ = classify_bags(res0, res1, Ys, class_alg=class_alg, ctx=ctx, rng=rng)
    diff = labels - est                      # test_one: label - est_label; 1 = false negative, -1 = false positive
    fn, fp = int(np.sum(diff == 1)), int(np.sum(diff == -1))
    n0, n1 = int(np.sum(labels == 0)), int(np.sum(labels != 0))
    n = labels.size
    with np.errstate(divide="ignore", invalid="ignore"):
        mer = (fp + fn) / n if n else float("nan")
        eer = float((np.float64(fp) / n0 + np.float64(fn) / n1) / 2)
    return mer, eer, fp, fn, n0, n1


test_classification.__test__ = False         # not a pytest test


def train_dual(Y0_train, Y1_train, H, H0, niter, eps=1e-4, verb=False, diag_var=False, ctx=None, rng=None, max_restarts=10):
    """`train_dual` examples/mil_util.jl:327-385: factorise the negative and the positive training matrix with `vbmf_dual!`
    (full_cov = true, at most floor(3200/H) randomly chosen columns each), restarting from a new random initialisation
    while the solution collapsed (||AHat|| + ||BHat|| < 1e-2), at most `max_restarts` times.  Returns (params0, params1)."""
    rng = rng or np.random.default_rng()
    maxM = int(3200 // H)
    out = []
    for Yt in (Y0_train, Y1_train):
        Yt = np.asarray(Yt, dtype=np.float64)
        M = Yt.shape[1]
        inds = rng.choice(M, size=min(maxM, M), replace=False)      # sample(1:M, min(maxM, M), replace = false), :344
        Ys = np.asfortranarray(Yt[:, inds])
        p = A.vbmf_dual_init(Ys, H, H0, rng=rng)
        nres, delta = 0, 1e-3
        while nres < max_restarts and delta < 1e-2:
            p = A.vbmf_dual_init(Ys, H, H0, rng=rng)
            A.vbmf_dual_(Ys, p, niter, eps=eps, diag_var=diag_var, full_cov=True, ctx=ctx, yhat=False)
            delta = _spectral(p.AHat) + _spectral(p.BHat)
            nres += 1
        if delta < 1e-2 and verb:
            print("Sensible result in samples factorization not achieved after %d retries!" % nres)
        out.append(p)
    return tuple(out)
