"""vbmf_b200_batched_plan (host only): which kernel of the batched vbls! path runs each problem of a batch."""
import ctypes

import numpy as np
import pytest

import vbmf_b200_loader

DENSE, SPARSE, DUAL, TRIAL = 0, 1, 2, 3


@pytest.fixture(scope="module")
def lib():
    vbmf_b200_loader.build()
    return vbmf_b200_loader.load()._lib.load()


def plan(lib, kind, L, H, Ms, full_cov=1, diag_var=0):
    M = np.ascontiguousarray(Ms, dtype=np.int64)
    out = np.full(M.size, -7, dtype=np.int32)
    rc = lib.vbmf_b200_batched_plan(kind, L, H, full_cov, diag_var, M.size, M.ctypes.data, out.ctypes.data)
    return rc, out


def fits_one_cta(kind, L, H, M):
    """The shared-memory footprint of the one-CTA-per-problem kernels (csrc/batched.cu) against their budgets."""
    if kind == DENSE:
        return (L * H + 2 * M * H + 3 * H * H + 2 * H) * 8 + 64 <= 200 * 1024
    work = 4 * (H * H + 98) + 2 if H <= 32 else H * (H + 1) + 3 * H
    return (L * H + 4 * M * H + 3 * H * H + H + 2 * L + 2 + work) * 8 + 64 <= 220 * 1024


@pytest.mark.parametrize("seed", range(6))
def test_plan_random_shapes(lib, seed):
    rng = np.random.default_rng(seed)
    for _ in range(40):
        kind = int(rng.integers(0, 4))
        H = int(rng.integers(1, (32 if kind == DENSE else 64) + 1))
        L = int(rng.integers(1, 400))
        Ms = np.sort(rng.integers(1, 5000, size=int(rng.integers(1, 30))))
        rc, cs = plan(lib, kind, L, H, Ms, full_cov=int(rng.integers(0, 2)), diag_var=int(rng.integers(0, 2)))
        assert rc == 0
        assert set(cs.tolist()) <= {0, 1, 2, 4, 8}
        for M, c in zip(Ms, cs):
            assert (c == 0) == fits_one_cta(kind, L, H, int(M)), (kind, L, H, M, c)
        # M ascending: the cluster size never decreases (a problem that fits comes first)
        assert np.all(np.diff(cs.astype(np.int64)) >= 0), (kind, L, H, Ms, cs)


def test_plan_known_shapes(lib):
    # the c2 shape: every bag of up to 301 columns fits; Musk2-sized bags (L = 166, up to 1044 columns) do not
    assert plan(lib, DUAL, 38, 20, [5, 40, 301])[1].tolist() == [0, 0, 0]
    rc, cs = plan(lib, DUAL, 166, 20, [1, 7, 300, 700, 1044])
    assert rc == 0 and cs[0] == 0 and cs[1] == 0 and np.all(cs[2:] >= 1)
    # L = 166, H = 64: one column fits one CTA, two do not (and get a cluster of one CTA)
    assert plan(lib, SPARSE, 166, 64, [1, 2])[1].tolist() == [0, 1]
    # the cluster never grows beyond 8 CTAs
    assert plan(lib, SPARSE, 38, 20, [10 ** 7])[1].tolist() == [8]
    assert plan(lib, DENSE, 166, 32, [267, 268])[1].tolist()[0] == 0


def test_plan_refuses_bad_arguments(lib):
    vb = vbmf_b200_loader.load()
    assert plan(lib, SPARSE, 38, 65, [5])[0] == -1
    assert "H <= 64" in lib.vbmf_b200_last_error().decode()
    assert plan(lib, DENSE, 38, 33, [5])[0] == -1
    assert "H <= 32" in lib.vbmf_b200_last_error().decode()
    assert plan(lib, SPARSE, 38, 64, [5])[0] == 0 and plan(lib, DENSE, 38, 32, [5])[0] == 0
    for args in ((4, 38, 20, [5]), (-1, 38, 20, [5]), (DUAL, 0, 20, [5]), (DUAL, 38, 0, [5]), (DUAL, 38, 20, [0]),
                 (DUAL, 38, 20, [5, -3])):
        assert plan(lib, *args)[0] == -1, args
    assert plan(lib, DUAL, 38, 20, [5], full_cov=2)[0] == -1
    assert plan(lib, DUAL, 38, 20, [5], diag_var=-1)[0] == -1
    assert lib.vbmf_b200_batched_plan(DUAL, 38, 20, 1, 0, 1, None, None) == -1
    assert lib.vbmf_b200_batched_plan(DUAL, 38, 20, 1, 0, -1, None, None) == -1
    assert lib.vbmf_b200_batched_plan(DUAL, 38, 20, 1, 0, 0, None, None) == 0
    with pytest.raises(vb.VBMFError, match="H <= 64"):
        vb._lib.check(plan(lib, TRIAL, 10, 100, [3])[0])
