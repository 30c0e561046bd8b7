"""Host-side mirror of VBMatrixFactorization.jl's exported API for the VB update loop, on top of the C ABI.

Same names, argument meaning and error behaviour as the reference (Julia `f!` becomes `f_` here):

    vbmf_init / vbmf_ / vbmf                       src/vbmf.jl:48,175,238
    vbmf_sparse_init / vbmf_sparse_ / vbmf_sparse  src/vbmf_sparse.jl:101,344,418
    vbmf_dual_init / vbmf_dual_ / vbmf_dual        src/vbmf_dual.jl:122,455,538
    updateA_, updateB_, updateCA_, updateCB_, updateSigma2_/updateSigma_, updateYHat_, updateAlpha00_ ...,
    lowerBound, lowerBoundTrimmed, copy, vbls_ (examples/mil_util.jl:179), vbls_batched_ / BatchedVbls and
    lowerBound_batched / lowerBoundTrimmed_batched (many small problems in one call)

Matrices are numpy arrays in Julia layout (Fortran order, Float64); labels are 1-based Int64.  The host keeps what the
reference keeps on the host: initialisation (RNG), argument checking and struct marshalling.  Everything inside the
while-loop runs on the GPU behind one ABI call with device-side convergence.  There is no CPU fallback.
"""
from __future__ import annotations

import copy as _copy
import ctypes as C

import numpy as np

from . import _lib as L_

__all__ = [
    "Context", "MultiContext", "default_context", "shard_columns",
    "vbmf_parameters", "vbmf_sparse_parameters", "vbmf_dual_parameters", "vbmf_trial_parameters", "vbmf_trial_init", "vbmf_trial_", "vbmf_trial",
    "vbmf_init", "vbmf_", "vbmf", "vbmf_sparse_init", "vbmf_sparse_", "vbmf_sparse", "vbmf_dual_init", "vbmf_dual_",
    "vbmf_dual", "updateA_", "updateB_", "updateCA_", "updateCB_", "updateSigma2_", "updateSigma_", "updateYHat_",
    "updateAlpha00_", "updateAlpha01_", "updateBeta00_", "updateBeta01_", "lowerBound", "lowerBoundTrimmed", "copy",
    "vbls_", "vbls_batched_", "BatchedVbls", "lowerBound_batched", "lowerBoundTrimmed_batched", "preprocess", "VBMFWarning", "create_log", "update_log_", "save_log", "load_log", "extract_params_", "VBMFError",
]

VBMFError = L_.VBMFError
_NORMS = {"spectral": L_.NORM_SPECTRAL, "frobenius": L_.NORM_FROBENIUS}


def _f(a, shape=None):
    a = np.asarray(a, dtype=np.float64)
    a = np.asfortranarray(a)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError("array of shape %s expected, got %s" % (tuple(shape), a.shape))
    return a


def _ptr(a):
    return a.ctypes.data if a is not None else None


def shard_columns(M, world, rank):
    """Column range [offset, offset+count) of Y owned by `rank` (contiguous, near-equal, multiples of 16 where possible)."""
    base, rem = divmod(M, world)
    counts = [base + (1 if r < rem else 0) for r in range(world)]
    off = sum(counts[:rank])
    return off, counts[rank]


# ----------------------------------------------------------------------------------------------------------- context
class Context:
    """One GPU (one rank): stream, NCCL communicator and the resident column shard of Y."""

    def __init__(self, device=0, rank=0, world=1, nccl_id=None, stream=None):
        self.lib = L_.load()
        self.rank, self.world, self.device = rank, world, device
        h = C.c_void_p()
        idbuf = (C.c_char * 128).from_buffer_copy(nccl_id) if nccl_id is not None else None
        L_.check(self.lib.vbmf_b200_ctx_create(device, rank, world, idbuf, C.c_void_p(stream) if stream else None, C.byref(h)))
        self.h = h
        self._key = None
        self.L = self.M = self.M_global = self.col_offset = 0

    @staticmethod
    def nccl_unique_id():
        buf = (C.c_char * 128)()
        L_.check(L_.load().vbmf_b200_nccl_unique_id(buf))
        return bytes(buf)

    def close(self):
        if getattr(self, "h", None):
            self.lib.vbmf_b200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def attach(self, Y, M_global=None, col_offset=0, force=True):
        """Upload this rank's L x M_local slice of Y.  Every call uploads: the library never guesses that a host array is
        unchanged (an in-place edit is invisible to any cheap fingerprint).  Residency is explicit instead: attach once, then
        pass Y=None to the drivers / step functions to run on the matrix already on the device (tests/mgpu_worker.py).
        `force` is accepted for backward compatibility and ignored."""
        Y = _f(Y)
        if Y.ndim != 2:
            raise ValueError("Y must be a matrix")
        Lr, M = Y.shape
        Mg = M if M_global is None else M_global
        L_.check(self.lib.vbmf_b200_attach_Y(self.h, _ptr(Y), Lr, M, max(Lr, 1), Mg, col_offset))
        self._Y_host = Y              # large uploads are asynchronous: the host buffer stays alive until the next attach
        self._key = ("host", Lr, M, Mg, col_offset)
        self.L, self.M, self.M_global, self.col_offset = Lr, M, Mg, col_offset

    def set_shape(self, Lr, M_local, M_global=None, col_offset=0):
        """Geometry only (no data): enough for the step functions that take no Y in the reference."""
        Mg = M_local if M_global is None else M_global
        L_.check(self.lib.vbmf_b200_set_shape(self.h, Lr, M_local, Mg, col_offset))
        self._key = None
        self.L, self.M, self.M_global, self.col_offset = Lr, M_local, Mg, col_offset

    def synth(self, Lr, M_local, M_global=None, col_offset=0, rank=8, noise=0.1, seed=20260101):
        Mg = M_local if M_global is None else M_global
        L_.check(self.lib.vbmf_b200_synth_Y(self.h, Lr, M_local, Mg, col_offset, rank, noise, seed))
        self._key = ("synth", Lr, M_local, Mg, col_offset, rank, noise, seed)
        self.L, self.M, self.M_global, self.col_offset = Lr, M_local, Mg, col_offset

    def preprocess(self, lam):
        """`preprocess(Y, lambda)` (src/util.jl:73-87) on the resident Y; returns the kept rows (1-based)."""
        rows = np.zeros(max(self.L, 1), dtype=np.int64)
        Ln = C.c_int64()
        L_.check(self.lib.vbmf_b200_preprocess_Y(self.h, float(lam), C.byref(Ln), rows.ctypes.data))
        self.L = Ln.value
        self._key = None
        return rows[:Ln.value].copy()

    def download_Y(self):
        Y = np.empty((self.L, self.M), order="F")
        L_.check(self.lib.vbmf_b200_download_Y(self.h, _ptr(Y), max(self.L, 1)))
        return Y

    def trYTY(self):
        v = C.c_double()
        L_.check(self.lib.vbmf_b200_trYTY(self.h, C.byref(v)))
        return v.value

    def sync(self):
        L_.check(self.lib.vbmf_b200_ctx_sync(self.h))

    def gemm_YtB(self, B):
        B = _f(B, (self.L, B.shape[1]))
        P = np.empty((self.M, B.shape[1]), order="F")
        L_.check(self.lib.vbmf_b200_gemm_YtB(self.h, _ptr(B), B.shape[1], _ptr(P)))
        return P

    def gemm_YA(self, A):
        A = _f(A, (self.M, A.shape[1]))
        Q = np.empty((self.L, A.shape[1]), order="F")
        L_.check(self.lib.vbmf_b200_gemm_YA(self.h, _ptr(A), A.shape[1], _ptr(Q)))
        return Q

    def peer_exchange(self):
        """True when updateB!'s exchange between the column shards runs through peer-mapped memory (own kernels over NVLink)."""
        return bool(self.lib.vbmf_b200_ctx_peer_exchange(self.h))

    def profile(self, enable=True, segments=False):
        L_.check(self.lib.vbmf_b200_ctx_profile(self.h, (3 if segments else 1) if enable else 0))

    def profile_read(self):
        a, b = C.c_double(), C.c_double()
        na, nb = C.c_int64(), C.c_int64()
        L_.check(self.lib.vbmf_b200_ctx_profile_read(self.h, C.byref(a), C.byref(na), C.byref(b), C.byref(nb)))
        ar, nar = C.c_double(), C.c_int64()
        L_.check(self.lib.vbmf_b200_ctx_profile_read_allreduce(self.h, C.byref(ar), C.byref(nar)))
        seg_ms, seg_n = (C.c_double * 32)(), (C.c_int64 * 32)()
        nseg = self.lib.vbmf_b200_ctx_profile_read_segments(self.h, seg_ms, seg_n, 32)
        names = ["start", "k1", "a_epilogue", "k2", "reduce_q", "exchange", "sigma_b", "b_epilogue", "b_reduce",
                 "wait_small", "wait_epilogue", "wait_reduce", "epi_fill", "epi_barrier", "epi_load", "epi_product", "epi_gram",
                 "epi_out", "red_local", "red_barrier", "red_final"]
        segs = {names[i]: seg_ms[i] / seg_n[i] for i in range(1, min(max(nseg, 0), len(names))) if seg_n[i] > 0}
        return {"k1_ms": a.value, "k1_launches": na.value, "k2_ms": b.value, "k2_launches": nb.value,
                "allreduce_ms": ar.value, "allreduce_launches": nar.value, "segments_ms": segs}


class MultiContext:
    """Several GPUs driven from THIS process (vbmf_b200_mctx): the reference is one Julia process making plain calls, so the
    column-sharded path must be reachable without one process per GPU.  Y and the parameter objects are the full-size host
    arrays; the library splits the columns over the devices, runs one host thread per device and gathers the results.
    Pass it as `ctx=` to vbmf_ / vbmf_sparse_ / vbmf_dual_ / vbmf_trial_ / lowerBound*."""

    def __init__(self, devices=None):
        self.lib = L_.load()
        h = C.c_void_p()
        if devices is None:
            L_.check(self.lib.vbmf_b200_mctx_create(0, None, C.byref(h)))
        else:
            devs = (C.c_int * len(devices))(*[int(x) for x in devices])
            L_.check(self.lib.vbmf_b200_mctx_create(len(devices), devs, C.byref(h)))
        self.h = h
        self.ndev = self.lib.vbmf_b200_mctx_ndev(h)
        self.world = 1          # one process: the sharding is internal
        self.L = self.M = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.vbmf_b200_mctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def attach(self, Y, **_):
        Y = _f(Y)
        if Y.ndim != 2:
            raise ValueError("Y must be a matrix")
        Lr, M = Y.shape
        L_.check(self.lib.vbmf_b200_mctx_attach_Y(self.h, _ptr(Y), Lr, M, max(Lr, 1)))
        self._Y_host = Y              # large uploads are asynchronous: the host buffer stays alive until the next attach
        self.L, self.M = Lr, M

    def synth(self, Lr, M, rank=8, noise=0.1, seed=20260101):
        L_.check(self.lib.vbmf_b200_mctx_synth_Y(self.h, Lr, M, rank, noise, seed))
        self.L, self.M = Lr, M

    def trYTY(self):
        v = C.c_double()
        L_.check(self.lib.vbmf_b200_mctx_trYTY(self.h, C.byref(v)))
        return v.value

    def shard(self, i):
        off, n = C.c_int64(), C.c_int64()
        L_.check(self.lib.vbmf_b200_mctx_shard(self.h, i, C.byref(off), C.byref(n)))
        return off.value, n.value

    def device_context(self, i):
        """Borrowed handle of device i's context (profiling)."""
        h = C.c_void_p()
        L_.check(self.lib.vbmf_b200_mctx_ctx(self.h, i, C.byref(h)))
        return h


_default_ctx = {}


def default_context(device=0):
    if device not in _default_ctx:
        _default_ctx[device] = Context(device=device)
    return _default_ctx[device]


def _ctx_for(Y, ctx):
    """Context for a call that takes Y.  Y=None: run on the matrix already resident in ctx.  On a sharded context
    (world > 1) a host Y must be this rank's shard: it is re-attached with the geometry (M_global, col_offset) the context
    already holds; a shard of a different shape cannot be placed and is refused instead of silently running with M_global = M_local."""
    ctx = ctx or default_context()
    if Y is not None:
        if ctx.world > 1:
            if ctx.M_global <= 0 or tuple(np.shape(Y)) != (ctx.L, ctx.M):
                raise VBMFError("sharded context (world=%d): pass Y=None after ctx.attach(Y_shard, M_global=..., col_offset=...), or a shard "
                                "of the attached shape %s (got %s)" % (ctx.world, (ctx.L, ctx.M), tuple(np.shape(Y))))
            ctx.attach(Y, M_global=ctx.M_global, col_offset=ctx.col_offset)
        else:
            ctx.attach(Y)
    return ctx


# ----------------------------------------------------------------------------------------------------------- parameter types
class _Params:
    _fields = ()

    def __repr__(self):
        return "%s(L=%d, M=%d, H=%d)" % (type(self).__name__, self.L, self.M, self.H)


class vbmf_parameters(_Params):
    """src/vbmf.jl:22-40"""
    kind = L_.DENSE


class vbmf_sparse_parameters(_Params):
    """src/vbmf_sparse.jl:47-90; SigmaATVec/invSigmaATVec are exposed block-wise (SigmaATVec_blocks, M x H x H) or None."""
    kind = L_.SPARSE


class vbmf_dual_parameters(_Params):
    """src/vbmf_dual.jl:59-112"""
    kind = L_.DUAL


class vbmf_trial_parameters(_Params):
    """src/vbmf_trial.jl:68-129 (unexported in the reference; used by examples/mil_util.jl)"""
    kind = L_.TRIAL


def copy(params_in):
    """Base.copy for the parameter types (src/vbmf.jl:80 is shallow; results are identical, a deep copy is made)."""
    return _copy.deepcopy(params_in)


def _labels(labels):
    return np.ascontiguousarray(np.asarray(labels if labels is not None else [], dtype=np.int64).reshape(-1))


def _mask(p):
    if p.H1 > 0 and p.labels.size > 0:
        p.AHat[p.labels - 1, p.H - p.H1:] = 0.0


def vbmf_init(Y, H, ca=1.0, cb=1.0, sigma2=1.0, H1=0, labels=None, rng=None):
    """src/vbmf.jl:48-73 (AHat drawn before BHat; YHat is produced lazily by updateYHat_)."""
    rng = rng or np.random.default_rng()
    Lr, M = Y.shape
    p = vbmf_parameters()
    p.L, p.M, p.H, p.H1 = Lr, M, int(H), int(H1)
    p.labels = _labels(labels)
    p.AHat = _f(rng.standard_normal((M, H)))
    _mask(p)
    p.BHat = _f(rng.standard_normal((Lr, H)))
    p.SigmaA = _f(np.zeros((H, H)))
    p.SigmaB = _f(np.zeros((H, H)))
    p.CA = _f(ca * np.eye(H))
    p.CB = _f(cb * np.eye(H))
    p.invCA = _f(np.linalg.inv(p.CA))
    p.invCB = _f(np.linalg.inv(p.CB))
    p.sigma2 = float(sigma2)
    p.YHat = None
    return p


def _sparse_common_init(p, Y, H, ca, cb, gamma0, delta0, sigma, eta0, zeta0, rng, trYTY):
    Lr, M = Y.shape
    p.L, p.M, p.H, p.MH = Lr, M, int(H), M * int(H)
    p.AHat = _f(rng.standard_normal((M, H)))
    p.SigmaATVec_blocks = None
    p.diagSigmaATVec = np.ones(M * H)
    p.SigmaA = _f(np.zeros((H, H)))
    p.BHat = _f(rng.standard_normal((Lr, H)))
    p.SigmaB = _f(np.zeros((H, H)))
    p.CB = cb * np.ones(H)
    p.gamma0, p.delta0 = float(gamma0), float(delta0)
    p.gamma = gamma0 + Lr / 2
    p.delta = delta0 * np.ones(H)
    p.sigmaHat = float(sigma)
    p.eta0, p.zeta0 = float(eta0), float(zeta0)
    p.eta = eta0 + Lr * M / 2
    p.zeta = float(zeta0)
    p.sigmaVecHat = sigma * np.ones(Lr)
    p.etaVec = (eta0 + M / 2) * np.ones(Lr)
    p.zetaVec = zeta0 * np.ones(Lr)
    p.YHat = None
    p.trYTY = float(np.sum(Y * Y)) if trYTY is None else float(trYTY)


def vbmf_sparse_init(Y, H, ca=1.0, alpha0=1e-10, beta0=1e-10, cb=1.0, gamma0=1e-10, delta0=1e-10, sigma=1.0,
                     eta0=1e-10, zeta0=1e-10, H1=0, labels=None, rng=None, trYTY=None):
    """src/vbmf_sparse.jl:101-153 (the eye(MH, MH) fields are never materialised)."""
    rng = rng or np.random.default_rng()
    p = vbmf_sparse_parameters()
    p.H1 = int(H1)
    p.labels = _labels(labels)
    _sparse_common_init(p, Y, H, ca, cb, gamma0, delta0, sigma, eta0, zeta0, rng, trYTY)
    _mask(p)
    p.ATVecHat = np.ascontiguousarray(p.AHat).reshape(p.MH).copy()
    p.CA = ca * np.ones(p.MH)
    p.alpha0, p.beta0 = float(alpha0), float(beta0)
    p.alpha = alpha0 + 0.5
    p.beta = beta0 * np.ones(p.MH)
    return p


def vbmf_dual_init(Y, H, H0, ca=1.0, alpha0=1e-10, beta0=1e-10, cb=1.0, gamma0=1e-10, delta0=1e-10, sigma=1.0,
                   eta0=1e-10, zeta0=1e-10, rng=None, trYTY=None):
    """src/vbmf_dual.jl:122-193"""
    if H < H0:
        raise VBMFError("H must be at least H0!")
    rng = rng or np.random.default_rng()
    p = vbmf_dual_parameters()
    p.H0, p.H1 = int(H0), int(H - H0)
    p.labels = _labels(None)
    _sparse_common_init(p, Y, H, ca, cb, gamma0, delta0, sigma, eta0, zeta0, rng, trYTY)
    M = p.M
    p.ATVecHat = np.ascontiguousarray(p.AHat).reshape(p.MH).copy()
    p.A0Hat = _f(p.AHat[:, :H0])
    p.A1Hat = _f(p.AHat[:, H0:])
    p.CA0 = ca * np.ones(M * p.H0)
    p.CA1 = ca * np.ones(M * p.H1)
    p.CA = ca * np.ones(p.MH)
    p.alpha00 = p.alpha01 = float(alpha0)
    p.beta00 = p.beta01 = float(beta0)
    p.alpha0 = p.alpha1 = alpha0 + 0.5
    p.beta0 = beta0 * np.ones(M * p.H0)
    p.beta1 = beta0 * np.ones(M * p.H1)
    p.alpha = np.array([p.alpha0, p.alpha1])
    p.beta = beta0 * np.ones(p.MH)
    return p


def vbmf_trial_init(Y, H, H0, M0, ca=1.0, alpha0=1e-10, beta0=1e-10, cb=1.0, gamma0=1e-10, delta0=1e-10, sigma=1.0,
                    eta0=1e-10, zeta0=1e-10, rng=None, trYTY=None):
    """src/vbmf_trial.jl:139-227"""
    if H < H0:
        raise VBMFError("H must be at least H0!")
    rng = rng or np.random.default_rng()
    p = vbmf_trial_parameters()
    p.H0, p.H1 = int(H0), int(H - H0)
    p.labels = _labels(None)
    _sparse_common_init(p, Y, H, ca, cb, gamma0, delta0, sigma, eta0, zeta0, rng, trYTY)
    M = p.M
    p.M0, p.M1 = int(M0), M - int(M0)
    p.ATVecHat = np.ascontiguousarray(p.AHat).reshape(p.MH).copy()
    p.A1Hat = _f(p.AHat[:, :H0])
    p.A2Hat = _f(p.AHat[:M0, H0:])
    p.A3Hat = _f(p.AHat[M0:, H0:])
    p.CA1, p.CA2, p.CA3 = ca * np.ones(M * p.H0), ca * np.ones(p.M0 * p.H1), ca * np.ones(p.M1 * p.H1)
    p.CA = ca * np.ones(p.MH)
    p.alpha01 = p.alpha02 = p.alpha03 = float(alpha0)
    p.beta01 = p.beta02 = p.beta03 = float(beta0)
    p.alpha1 = p.alpha2 = p.alpha3 = alpha0 + 0.5
    p.beta1, p.beta2, p.beta3 = beta0 * np.ones(M * p.H0), beta0 * np.ones(p.M0 * p.H1), beta0 * np.ones(p.M1 * p.H1)
    p.alpha = np.array([p.alpha1, p.alpha2, p.alpha3])
    p.beta = beta0 * np.ones(p.MH)
    return p


# ----------------------------------------------------------------------------------------------------------- marshalling
def _ensure(p, name, shape, fortran=True):
    a = getattr(p, name, None)
    if a is None or a.shape != tuple(shape) or a.dtype != np.float64 or not (a.flags.f_contiguous if fortran else a.flags.c_contiguous):
        a = (_f(a, shape) if a is not None else (np.zeros(shape, order="F")))
        setattr(p, name, a)
    return a


def _dense_struct(p, want_yhat):
    H = p.H
    st = L_.DenseState()
    st.L, st.M, st.H, st.H1 = p.L, p.M, H, p.H1
    p.labels = _labels(p.labels)
    st.n_labels = p.labels.size
    st.labels = p.labels.ctypes.data if p.labels.size else None
    st.AHat = _ptr(_ensure(p, "AHat", (p.M, H)))
    st.BHat = _ptr(_ensure(p, "BHat", (p.L, H)))
    for f in ("SigmaA", "SigmaB", "CA", "CB", "invCA", "invCB"):
        setattr(st, f, _ptr(_ensure(p, f, (H, H))))
    st.sigma2 = p.sigma2
    if want_yhat:
        p.YHat = np.empty((p.L, p.M), order="F")
        st.YHat = _ptr(p.YHat)
    return st


def _sparse_fill(st, p, want_yhat, want_blocks):
    H, M, Lr = p.H, p.M, p.L
    st.L, st.M, st.H, st.MH = Lr, M, H, M * H
    st.AHat = _ptr(_ensure(p, "AHat", (M, H)))
    p.ATVecHat = np.ascontiguousarray(p.AHat).reshape(M * H) if getattr(p, "ATVecHat", None) is None else np.ascontiguousarray(p.ATVecHat, dtype=np.float64)
    st.ATVecHat = _ptr(p.ATVecHat)
    for f, n in (("diagSigmaATVec", M * H), ("CA", M * H), ("beta", M * H), ("CB", H), ("delta", H), ("sigmaVecHat", Lr),
                 ("etaVec", Lr), ("zetaVec", Lr)):
        a = np.ascontiguousarray(getattr(p, f), dtype=np.float64).reshape(n)
        setattr(p, f, a)
        setattr(st, f, _ptr(a))
    for f in ("SigmaA", "SigmaB"):
        setattr(st, f, _ptr(_ensure(p, f, (H, H))))
    st.BHat = _ptr(_ensure(p, "BHat", (Lr, H)))
    if want_blocks:
        if getattr(p, "SigmaATVec_blocks", None) is None or p.SigmaATVec_blocks.shape != (M, H, H):
            p.SigmaATVec_blocks = np.zeros((M, H, H))
        st.SigmaATVec_blocks = _ptr(p.SigmaATVec_blocks)
    for f in ("gamma0", "delta0", "gamma", "sigmaHat", "eta0", "zeta0", "eta", "zeta", "trYTY"):
        setattr(st, f, float(getattr(p, f)))
    if want_yhat:
        p.YHat = np.empty((Lr, M), order="F")
        st.YHat = _ptr(p.YHat)


def _sparse_struct(p, want_yhat, want_blocks):
    st = L_.SparseState()
    _sparse_fill(st, p, want_yhat, want_blocks)
    st.H1 = p.H1
    p.labels = _labels(p.labels)
    st.n_labels = p.labels.size
    st.labels = p.labels.ctypes.data if p.labels.size else None
    st.alpha0, st.beta0, st.alpha = p.alpha0, p.beta0, p.alpha
    return st


def _dual_struct(p, want_yhat, want_blocks):
    st = L_.DualState()
    _sparse_fill(st, p, want_yhat, want_blocks)
    M = p.M
    st.H0, st.H1 = p.H0, p.H1
    st.A0Hat = _ptr(_ensure(p, "A0Hat", (M, p.H0)))
    st.A1Hat = _ptr(_ensure(p, "A1Hat", (M, p.H1)))
    for f, n in (("CA0", M * p.H0), ("CA1", M * p.H1), ("beta0", M * p.H0), ("beta1", M * p.H1), ("alpha", 2)):
        a = np.ascontiguousarray(getattr(p, f), dtype=np.float64).reshape(n)
        setattr(p, f, a)
        setattr(st, f, _ptr(a))
    for f in ("alpha00", "beta00", "alpha0", "alpha01", "beta01", "alpha1"):
        setattr(st, f, float(getattr(p, f)))
    return st


def _trial_struct(p, want_yhat, want_blocks, m2_local=None):
    """m2_local: number of this shard's rows that belong to group 2 (global index <= M0); defaults to the unsharded M0."""
    st = L_.TrialState()
    _sparse_fill(st, p, want_yhat, want_blocks)
    M = p.M
    m2 = p.M0 if m2_local is None else m2_local
    m2 = max(0, min(int(m2), M))
    st.M0, st.M1, st.H0, st.H1 = p.M0, p.M1, p.H0, p.H1
    st.A1Hat = _ptr(_ensure(p, "A1Hat", (M, p.H0)))
    st.A2Hat = _ptr(_ensure(p, "A2Hat", (m2, p.H1)))
    st.A3Hat = _ptr(_ensure(p, "A3Hat", (M - m2, p.H1)))
    for f, n in (("CA1", M * p.H0), ("CA2", m2 * p.H1), ("CA3", (M - m2) * p.H1), ("beta1", M * p.H0), ("beta2", m2 * p.H1),
                 ("beta3", (M - m2) * p.H1), ("alpha", 3)):
        a = np.ascontiguousarray(getattr(p, f), dtype=np.float64).reshape(-1)
        if a.size != n:
            a = np.zeros(n)
        setattr(p, f, a)
        setattr(st, f, _ptr(a))
    for f in ("alpha01", "beta01", "alpha1", "alpha02", "beta02", "alpha2", "alpha03", "beta03", "alpha3"):
        setattr(st, f, float(getattr(p, f)))
    return st


def _readback(p, st):
    if p.kind == L_.DENSE:
        p.sigma2 = st.sigma2
        return
    for f in ("sigmaHat", "zeta", "eta"):
        setattr(p, f, getattr(st, f))
    if p.kind == L_.DUAL:
        for f in ("alpha00", "beta00", "alpha01", "beta01", "alpha0", "alpha1"):
            setattr(p, f, getattr(st, f))
    if p.kind == L_.TRIAL:
        for f in ("alpha01", "beta01", "alpha1", "alpha02", "beta02", "alpha2", "alpha03", "beta03", "alpha3"):
            setattr(p, f, getattr(st, f))


def _struct(p, want_yhat=False, want_blocks=False):
    if p.kind == L_.DENSE:
        return _dense_struct(p, want_yhat)
    if p.kind == L_.SPARSE:
        return _sparse_struct(p, want_yhat, want_blocks)
    if p.kind == L_.TRIAL:
        return _trial_struct(p, want_yhat, want_blocks, getattr(p, "_m2_local", None))
    return _dual_struct(p, want_yhat, want_blocks)


_UP = {L_.DENSE: "vbmf_b200_dense_upload", L_.SPARSE: "vbmf_b200_sparse_upload", L_.DUAL: "vbmf_b200_dual_upload",
       L_.TRIAL: "vbmf_b200_trial_upload"}
_DOWN = {L_.DENSE: "vbmf_b200_dense_download", L_.SPARSE: "vbmf_b200_sparse_download", L_.DUAL: "vbmf_b200_dual_download",
         L_.TRIAL: "vbmf_b200_trial_download"}


class Solver:
    """Device-resident state of one problem (vbmf_b200_solver): upload once, step / run many times, download."""

    def __init__(self, ctx, params, keep_blocks=False):
        if isinstance(ctx, MultiContext):
            raise VBMFError("step-level calls, logging and vbls_ hold device-resident state of ONE context: use a single-device Context "
                            "(the multi-device context offers the whole-loop drivers and lowerBound)")
        self.ctx, self.lib = ctx, ctx.lib
        p = params
        if (p.L, p.M) != (ctx.L, ctx.M):
            raise VBMFError("params are %d x %d but the attached Y is %d x %d" % (p.L, p.M, ctx.L, ctx.M))
        split = p.H0 if p.kind in (L_.DUAL, L_.TRIAL) else p.H1
        labels = _labels(getattr(p, "labels", None))
        h = C.c_void_p()
        if p.kind == L_.TRIAL:
            L_.check(self.lib.vbmf_b200_solver_create_trial(ctx.h, p.H, p.H0, p.M0, 1 if keep_blocks else 0, C.byref(h)))
        else:
            L_.check(self.lib.vbmf_b200_solver_create(ctx.h, p.kind, p.H, split, labels.size,
                                                      labels.ctypes.data if labels.size else None,
                                                      1 if keep_blocks else 0, C.byref(h)))
        self.h, self.kind, self.keep_blocks = h, p.kind, keep_blocks

    def upload(self, p):
        st = _struct(p, False, self.keep_blocks)
        L_.check(getattr(self.lib, _UP[self.kind])(self.h, C.byref(st)))

    def download(self, p, want_yhat=False):
        st = _struct(p, want_yhat, self.keep_blocks)
        L_.check(getattr(self.lib, _DOWN[self.kind])(self.h, C.byref(st)))
        _readback(p, st)

    def step(self, step, flags=0):
        L_.check(self.lib.vbmf_b200_solver_step(self.h, step, flags))

    def run(self, niter, eps=1e-6, flags=0, norm="spectral"):
        it, d = C.c_int64(), C.c_double()
        self.failed = _not_pd(L_.check(self.lib.vbmf_b200_solver_run(self.h, int(niter), float(eps), flags, _NORMS[norm], C.byref(it), C.byref(d)),
                                       allow=(-2,))) == -2
        return it.value, d.value

    def lower_bound(self, trim=0.0, trimmed=False):
        v = C.c_double()
        L_.check(self.lib.vbmf_b200_solver_lower_bound(self.h, float(trim), 1 if trimmed else 0, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "h", None):
            self.lib.vbmf_b200_solver_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class VBMFWarning(RuntimeWarning):
    """A posterior precision matrix was not positive definite: NaN was written and the loop ended (ABI return code -2)."""


def _not_pd(rc, params=None):
    """Return code -2: the reference's LU `inv` would return garbage (or throw SingularException); here the state carries NaN,
    `params.failed` is set and a VBMFWarning names the cause.  Nothing is swallowed silently."""
    if params is not None:
        params.failed = rc == -2
    if rc == -2:
        import warnings
        msg = (L_.load().vbmf_b200_last_error() or b"").decode("utf-8", "replace")
        warnings.warn(VBMFWarning(msg or "a posterior precision matrix was not positive definite"), stacklevel=3)
    return rc


def _flags(diag_var=False, full_cov=False, est_cb=False, est_priors=False, est_covs=False, est_var=False):
    return ((L_.DIAG_VAR if diag_var else 0) | (L_.FULL_COV if full_cov else 0) | (L_.EST_CB if est_cb else 0) |
            (L_.EST_PRIORS if est_priors else 0) | (L_.EST_COVS if est_covs else 0) | (L_.EST_VAR if est_var else 0))


def _run_call(ctx, name):
    """The one-call drop-in of the single-device context or its multi-device twin."""
    return getattr(ctx.lib, ("vbmf_b200_mctx_" if isinstance(ctx, MultiContext) else "vbmf_b200_") + name)


def _verb(verb, it, d):
    if verb:
        print("Factorization finished after ", it, " iterations, eps = ", d)


# ----------------------------------------------------------------------------------------------------------- drivers
def vbmf_(Y, params, niter, eps=1e-6, est_covs=False, est_var=False, verb=False, norm="spectral", ctx=None, yhat=True,
          logdir="", desc=""):
    """`vbmf!` src/vbmf.jl:175-231: mutates params, returns params.  yhat=False skips the final L x M updateYHat!.
    logdir != "" logs every field after every iteration (create_log / update_log! / save_log)."""
    if logdir:
        it, d, params.log = _run_logged(Y, params, niter, eps, _flags(est_covs=est_covs, est_var=est_var), norm, ctx, logdir, desc)
        params.iterations, params.d = it, d
        _verb(verb, it, d)
        return params
    ctx = _ctx_for(Y, ctx)
    st = _dense_struct(params, yhat)
    it, d = C.c_int64(), C.c_double()
    _not_pd(L_.check(_run_call(ctx, "dense_run")(ctx.h, C.byref(st), int(niter), float(eps), int(est_covs), int(est_var), _NORMS[norm],
                                         C.byref(it), C.byref(d)), allow=(-2,)), params)
    _readback(params, st)
    params.iterations, params.d = it.value, d.value
    _verb(verb, it.value, d.value)
    return params


def vbmf(Y, params_in, niter, **kw):
    """src/vbmf.jl:238-248: copies params_in, returns the new params."""
    return vbmf_(Y, copy(params_in), niter, **kw)


def vbmf_sparse_(Y, params, niter, eps=1e-6, diag_var=False, full_cov=False, verb=False, est_cb=True, norm="spectral",
                 ctx=None, keep_blocks=False, yhat=True, logdir="", desc=""):
    """`vbmf_sparse!` src/vbmf_sparse.jl:344-410: mutates params, returns d."""
    if logdir:
        it, d, params.log = _run_logged(Y, params, niter, eps, _flags(diag_var=diag_var, full_cov=full_cov, est_cb=est_cb), norm, ctx,
                                        logdir, desc, keep_blocks)
        params.iterations = it
        _verb(verb, it, d)
        return d
    ctx = _ctx_for(Y, ctx)
    st = _sparse_struct(params, yhat, keep_blocks)
    it, d = C.c_int64(), C.c_double()
    _not_pd(L_.check(_run_call(ctx, "sparse_run")(ctx.h, C.byref(st), int(niter), float(eps), int(diag_var), int(full_cov), int(est_cb),
                                          _NORMS[norm], C.byref(it), C.byref(d)), allow=(-2,)), params)
    _readback(params, st)
    params.AHat = _f(params.AHat)
    params.iterations = it.value
    _verb(verb, it.value, d.value)
    return d.value


def vbmf_sparse(Y, params_in, niter, **kw):
    """src/vbmf_sparse.jl:418-428 -> (params, d)"""
    p = copy(params_in)
    d = vbmf_sparse_(Y, p, niter, **kw)
    return p, d


def vbmf_dual_(Y, params, niter, eps=1e-6, diag_var=False, full_cov=False, verb=False, est_priors=True, est_cb=True,
               norm="spectral", ctx=None, keep_blocks=False, yhat=True, logdir="", desc=""):
    """`vbmf_dual!` src/vbmf_dual.jl:455-530: mutates params, returns d."""
    if logdir:
        it, d, params.log = _run_logged(Y, params, niter, eps, _flags(diag_var=diag_var, full_cov=full_cov, est_cb=est_cb,
                                                                      est_priors=est_priors), norm, ctx, logdir, desc, keep_blocks)
        params.iterations = it
        _verb(verb, it, d)
        return d
    ctx = _ctx_for(Y, ctx)
    st = _dual_struct(params, yhat, keep_blocks)
    it, d = C.c_int64(), C.c_double()
    _not_pd(L_.check(_run_call(ctx, "dual_run")(ctx.h, C.byref(st), int(niter), float(eps), int(diag_var), int(full_cov), int(est_priors),
                                        int(est_cb), _NORMS[norm], C.byref(it), C.byref(d)), allow=(-2,)), params)
    _readback(params, st)
    params.iterations = it.value
    _verb(verb, it.value, d.value)
    return d.value


def vbmf_dual(Y, params_in, niter, **kw):
    """src/vbmf_dual.jl:538-549 -> (params, d)"""
    p = copy(params_in)
    d = vbmf_dual_(Y, p, niter, **kw)
    return p, d


def vbmf_trial_(Y, params, niter, eps=1e-6, diag_var=False, full_cov=False, verb=False, est_priors=True, est_cb=True,
                norm="spectral", ctx=None, keep_blocks=False, yhat=True, logdir="", desc=""):
    """`vbmf_trial!` src/vbmf_trial.jl:528-604: mutates params, returns d."""
    if logdir:
        it, d, params.log = _run_logged(Y, params, niter, eps, _flags(diag_var=diag_var, full_cov=full_cov, est_cb=est_cb,
                                                                      est_priors=est_priors), norm, ctx, logdir, desc, keep_blocks)
        params.iterations = it
        _verb(verb, it, d)
        return d
    ctx = _ctx_for(Y, ctx)
    st = _trial_struct(params, yhat, keep_blocks, getattr(params, "_m2_local", None))
    it, d = C.c_int64(), C.c_double()
    _not_pd(L_.check(_run_call(ctx, "trial_run")(ctx.h, C.byref(st), int(niter), float(eps), int(diag_var), int(full_cov), int(est_priors),
                                         int(est_cb), _NORMS[norm], C.byref(it), C.byref(d)), allow=(-2,)), params)
    _readback(params, st)
    params.iterations = it.value
    _verb(verb, it.value, d.value)
    return d.value


def vbmf_trial(Y, params_in, niter, **kw):
    """src/vbmf_trial.jl:612-623 -> (params, d)"""
    p = copy(params_in)
    d = vbmf_trial_(Y, p, niter, **kw)
    return p, d


# ----------------------------------------------------------------------------------------------------------- step functions
def _shape_for(params, ctx):
    """Y-less steps (updateCA!(params), ...): make sure the context's geometry matches the params."""
    ctx = ctx or default_context()
    if (ctx.L, ctx.M) != (params.L, params.M):
        ctx.set_shape(params.L, params.M)
    return ctx


def _a_mismatch(params):
    """True when AHat and ATVecHat (= vec(AHat')) of a sparse / dual / trial params object disagree, e.g. after
    `params.AHat = X` (examples/toy_data.jl:54).  The reference keeps two host copies: updateB!/updateSigma!/lowerBound read
    AHat, updateCA!/lowerBound read ATVecHat.  The device holds ONE factor, so the step functions pick the copy their
    reference counterpart reads and leave the other host copy untouched."""
    if params.kind == L_.DENSE or getattr(params, "ATVecHat", None) is None:
        return False
    return not np.array_equal(np.ascontiguousarray(params.AHat).reshape(-1), np.asarray(params.ATVecHat).reshape(-1))


def _one_step(Y, params, step, flags=0, ctx=None, want_yhat=False):
    ctx = _ctx_for(Y, ctx) if Y is not None else _shape_for(params, ctx)
    keep = None
    if _a_mismatch(params):
        if step == L_.STEP_UPDATE_CA:            # updateCA! reads ATVecHat and leaves AHat alone (src/vbmf_sparse.jl:284-288)
            keep = ("AHat", params.AHat.copy())
            params.AHat = _f(np.asarray(params.ATVecHat).reshape(params.M, params.H))
        elif step != L_.STEP_UPDATE_A:           # updateB! / updateSigma! / updateYHat! read AHat and leave ATVecHat alone
            keep = ("ATVecHat", np.array(params.ATVecHat))
            params.ATVecHat = np.ascontiguousarray(params.AHat).reshape(-1).copy()
    s = Solver(ctx, params, keep_blocks=bool(flags & L_.FULL_COV) and getattr(params, "SigmaATVec_blocks", None) is not None)
    try:
        s.upload(params)
        if step is not None:
            s.step(step, flags)
        s.download(params, want_yhat=want_yhat)
    finally:
        s.close()
        if keep is not None:
            setattr(params, keep[0], keep[1])


def updateA_(Y, params, full_cov=False, diag_var=False, ctx=None):
    """updateA! src/vbmf.jl:95, src/vbmf_sparse.jl:176, src/vbmf_dual.jl:216"""
    _one_step(Y, params, L_.STEP_UPDATE_A, _flags(diag_var=diag_var, full_cov=full_cov), ctx)


def updateB_(Y, params, diag_var=False, ctx=None):
    """updateB! src/vbmf.jl:109, src/vbmf_sparse.jl:254, src/vbmf_dual.jl:292"""
    _one_step(Y, params, L_.STEP_UPDATE_B, _flags(diag_var=diag_var), ctx)


def updateCA_(params, ctx=None):
    """updateCA! src/vbmf.jl:129, src/vbmf_sparse.jl:284, src/vbmf_dual.jl:322"""
    _one_step(None, params, L_.STEP_UPDATE_CA, 0, ctx)


def updateCB_(params, ctx=None):
    """updateCB! src/vbmf.jl:141, src/vbmf_sparse.jl:295, src/vbmf_dual.jl:358"""
    _one_step(None, params, L_.STEP_UPDATE_CB, 0, ctx)


def updateSigma2_(Y, params, ctx=None):
    """updateSigma2! src/vbmf.jl:153"""
    _one_step(Y, params, L_.STEP_UPDATE_SIGMA, 0, ctx)


def updateSigma_(Y, params, diag_var=False, ctx=None):
    """updateSigma! src/vbmf_sparse.jl:307, src/vbmf_dual.jl:370"""
    _one_step(Y, params, L_.STEP_UPDATE_SIGMA, _flags(diag_var=diag_var), ctx)


def updateYHat_(params, ctx=None):
    """updateYHat! src/vbmf.jl:120"""
    _one_step(None, params, None, 0, ctx, want_yhat=True)


def _prior_step(params, step, ctx):
    ctx = _shape_for(params, ctx)
    s = Solver(ctx, params)
    try:
        s.upload(params)
        s.step(step, 0)          # the library sums the current CA / beta vectors itself, the state stays untouched
        s.download(params)
    finally:
        s.close()


def updateAlpha00_(params, ctx=None):
    _prior_step(params, L_.STEP_UPDATE_ALPHA00, ctx)


def updateAlpha01_(params, ctx=None):
    _prior_step(params, L_.STEP_UPDATE_ALPHA01, ctx)


def updateBeta00_(params, ctx=None):
    _prior_step(params, L_.STEP_UPDATE_BETA00, ctx)


def updateBeta01_(params, ctx=None):
    _prior_step(params, L_.STEP_UPDATE_BETA01, ctx)


def lowerBound(Y, params, ctx=None):
    """lowerBound src/vbmf_sparse.jl:435, src/vbmf_dual.jl:556"""
    if _a_mismatch(params):
        raise VBMFError("lowerBound: params.AHat and params.ATVecHat disagree (the reference would mix the two copies); set both")
    ctx = _ctx_for(Y, ctx)
    if isinstance(ctx, MultiContext):
        return _multi_lower_bound(ctx, params, 0.0, False)
    s = Solver(ctx, params)
    try:
        s.upload(params)
        return s.lower_bound(0.0, False)
    finally:
        s.close()


def lowerBoundTrimmed(Y, params, trim=1e-1, ctx=None):
    """lowerBoundTrimmed src/vbmf_sparse.jl:478, src/vbmf_dual.jl:606"""
    if _a_mismatch(params):
        raise VBMFError("lowerBoundTrimmed: params.AHat and params.ATVecHat disagree (the reference would mix the two copies); set both")
    ctx = _ctx_for(Y, ctx)
    if isinstance(ctx, MultiContext):
        return _multi_lower_bound(ctx, params, trim, True)
    s = Solver(ctx, params)
    try:
        s.upload(params)
        return s.lower_bound(trim, True)
    finally:
        s.close()


def _multi_lower_bound(ctx, params, trim, trimmed):
    if params.kind == L_.DENSE:
        raise VBMFError("the dense solver has no lowerBound (the reference defines none)")
    st = _struct(params, False, False)
    v = C.c_double()
    L_.check(ctx.lib.vbmf_b200_mctx_lower_bound(ctx.h, params.kind, C.byref(st), float(trim), 1 if trimmed else 0, C.byref(v)))
    return v.value


def vbls_(Y, params, niter, diag_var=False, full_cov=False, ctx=None):
    """`vbls!` examples/mil_util.jl:179-203: niter x (updateA!, updateCA!, updateSigma*!) with BHat fixed; state stays resident."""
    ctx = _ctx_for(Y, ctx)
    fl = _flags(diag_var=diag_var, full_cov=full_cov)
    s = Solver(ctx, params)
    try:
        s.upload(params)
        for _ in range(niter):
            s.step(L_.STEP_UPDATE_A, fl)
            s.step(L_.STEP_UPDATE_CA, fl)
            s.step(L_.STEP_UPDATE_SIGMA, fl)
        s.download(params, want_yhat=True)
    finally:
        s.close()
    return params.AHat


class BatchedVbls:
    """Marshalled batch for `vbmf_b200_batched_vbls`: the per-problem state structs and pointer tables are built once here
    (pure Python/ctypes work, ~70 us per problem), `run` is then the bare C-ABI call on the host arrays the structs point
    at, and `readback` copies the scalar results back into the Python parameter objects.  A Julia caller pays none of the
    Python cost; `bench.py --workload c2` times `run` and reports the marshalling separately."""

    def __init__(self, Ys, params_list, ctx=None, yhat=True, keep_blocks=False):
        self.ctx = ctx or default_context()
        self.params = list(params_list)
        self.n = len(self.params)
        if self.n == 0:
            return
        self.kind = self.params[0].kind
        if any(p.kind != self.kind for p in self.params):
            raise VBMFError("vbls_batched_ needs a homogeneous list of parameters (all dense, all sparse, all dual or all trial)")
        self.Ys = [_f(Y) for Y in Ys]
        self.structs = [_struct(p, yhat, keep_blocks) for p in self.params]
        self.yp = (L_.p_f64 * self.n)(*[_ptr(Y) for Y in self.Ys])
        self.sp = (C.c_void_p * self.n)(*[C.addressof(st) for st in self.structs])

    def run(self, niter, full_cov=False, diag_var=False):
        if self.n == 0:
            return 0
        rc = _not_pd(L_.check(self.ctx.lib.vbmf_b200_batched_vbls(self.ctx.h, self.kind, self.n, self.yp, self.sp, int(niter),
                                                                  (L_.FULL_COV if full_cov else 0) | (L_.DIAG_VAR if diag_var else 0)),
                              allow=(-2,)))
        self.failed = rc == -2
        return rc

    def readback(self):
        for p, st in zip(self.params, self.structs):
            _readback(p, st)
        return [p.AHat for p in self.params]

    def lower_bound(self, trim=None):
        """lowerBound (trim = None) or lowerBoundTrimmed(trim) of every problem in one C-ABI call
        (`vbmf_b200_batched_lower_bound`) on the structs this object holds: after `run` they already point at the vbls
        results, so nothing is marshalled again.  Returns a float64 array, one bound per problem."""
        out = np.zeros(self.n)
        if self.n == 0:
            return out
        if isinstance(self.ctx, MultiContext):
            raise VBMFError("the batched lowerBound runs on one device: pass a single-device Context, not a MultiContext")
        if self.kind == L_.DENSE:
            raise VBMFError("the dense solver has no lowerBound (the reference defines none)")
        for i, p in enumerate(self.params):
            if _a_mismatch(p):
                raise VBMFError("lowerBound: params.AHat and params.ATVecHat of problem %d disagree (the reference would mix the two "
                                "copies); set both" % i)
        L_.check(self.ctx.lib.vbmf_b200_batched_lower_bound(self.ctx.h, self.kind, self.n, self.yp, self.sp,
                                                            0.0 if trim is None else float(trim), 0 if trim is None else 1,
                                                            out.ctypes.data))
        return out


def vbls_batched_(Ys, params_list, niter, full_cov=False, diag_var=False, ctx=None, yhat=True, keep_blocks=False):
    """`vbls!` (examples/mil_util.jl:179-203) for many problems in ONE C-ABI call (one CTA per problem; problems too large
    for one CTA's shared memory get a thread-block cluster each): the MIL classification pattern, classify(...; class_alg =
    "dual") runs it for every test bag and class model.  All params must be of one type (vbmf_parameters,
    vbmf_sparse_parameters, vbmf_dual_parameters or vbmf_trial_parameters - the four branches of vbls!) with the same L, H
    (and H0); M (and M0) may differ per problem."""
    batch = BatchedVbls(Ys, params_list, ctx=ctx, yhat=yhat, keep_blocks=keep_blocks)
    batch.run(niter, full_cov=full_cov, diag_var=diag_var)
    return batch.readback()


def lowerBound_batched(Ys, params_list, ctx=None):
    """`lowerBound` (src/vbmf_sparse.jl:435, src/vbmf_dual.jl:556, src/vbmf_trial.jl:630) of many problems in ONE C-ABI call:
    the ELBO of every (bag, class model) pair of a MIL test set.  Same grouping rules as `vbls_batched_` (one parameter type
    among sparse / dual / trial, the same L, H and H0; H <= 64), one device, no attached Y needed.  Returns a float64 array."""
    return BatchedVbls(Ys, params_list, ctx=ctx, yhat=False).lower_bound()


def lowerBoundTrimmed_batched(Ys, params_list, trim=1e-1, ctx=None):
    """`lowerBoundTrimmed` (src/vbmf_sparse.jl:478, src/vbmf_dual.jl:606, src/vbmf_trial.jl:687) of many problems in one
    call, as `lowerBound_batched`."""
    return BatchedVbls(Ys, params_list, ctx=ctx, yhat=False).lower_bound(float(trim))


def preprocess(Y, lam, verb=False, ctx=None):
    """`preprocess(Y, lambda; verb)` src/util.jl:73-87: returns the scaled matrix with near-constant rows removed, times lambda.
    The result also stays resident on the device (ctx): solvers called with Y=None run on it."""
    ctx = ctx or default_context()
    Y = _f(Y)
    ctx.attach(Y)
    L0 = ctx.L
    rows = ctx.preprocess(lam)
    if verb:
        print("Original problem size: %d rows, %d rows not relevant and are not used." % (L0, L0 - rows.size))
    return ctx.download_Y()       # the processed matrix also stays resident: pass Y=None to run on it without another upload


# ----------------------------------------------------------------------------------------------------------- trajectory logging (N4)
_LOG_SKIP = ("YHat", "SigmaATVec_blocks", "iterations", "d", "kind", "log", "failed")


def _log_fields(params):
    return [k for k, v in vars(params).items() if k not in _LOG_SKIP and v is not None and not k.startswith("_")]


def create_log(params):
    """`create_log` src/data_manip.jl:6-25: one entry per params field; scalars become 1-element vectors.
    YHat and the (MH)^2 covariance are not logged (the reference logs a stale YHat, SURVEY section 4)."""
    log = {}
    for k in _log_fields(params):
        v = getattr(params, k)
        if isinstance(v, (dict, list, tuple, str)) or not np.issubdtype(np.asarray(v).dtype, np.number):
            continue                      # only numeric fields are logged (src/data_manip.jl:10-22 handles Array / Number)
        log[k] = [np.array(v, dtype=np.float64 if not isinstance(v, (int, np.integer)) else np.int64)]
    return log


def update_log_(log, params):
    """`update_log!` src/data_manip.jl:32-45: append the current value of every field (new last dimension)."""
    for k in log:
        v = getattr(params, k)
        log[k].append(np.array(v, dtype=log[k][0].dtype))


def _stack(log):
    return {k: (np.stack(v, axis=-1) if v[0].ndim else np.array(v)) for k, v in log.items()}


def save_log(log, Y, priors, logdir, desc=""):
    """`save_log` src/data_manip.jl:53-66: <logdir>/<desc>/log.npz and inputs.npz (NumPy containers instead of JLD)."""
    import datetime
    import os
    desc = desc or datetime.datetime.now().strftime("%Y%m%d_%H%M%S")
    d = os.path.join(logdir, desc)
    os.makedirs(d, exist_ok=True)
    np.savez_compressed(os.path.join(d, "log.npz"), **_stack(log))
    np.savez_compressed(os.path.join(d, "inputs.npz"), Y=np.asarray(Y), **{"prior_" + k: v for k, v in (priors or {}).items()})
    return d


def load_log(path):
    """`load_log` src/data_manip.jl:74-89 -> (log dict of stacked arrays, Y)."""
    import os
    lg = np.load(os.path.join(path, "log.npz"))
    Y = np.load(os.path.join(path, "inputs.npz"))["Y"]
    return {k: lg[k] for k in lg.files}, Y


def extract_params_(log, params, i):
    """`extract_params!` src/data_manip.jl:96-118: overwrite params with slice i (0 = initial state) of a stacked log."""
    for k, v in log.items():
        if hasattr(params, k):
            cur = getattr(params, k)
            val = v[..., i]
            setattr(params, k, type(cur)(val) if np.ndim(cur) == 0 else np.array(val, order="F" if np.ndim(val) == 2 else "C"))
    return params


def _run_logged(Y, params, niter, eps, flags, norm, ctx, logdir, desc, keep_blocks=False):
    """The reference's loop with update_log! after every iteration (src/vbmf.jl:206-208): the state stays resident, one
    device iteration at a time, small fields are downloaded in between."""
    ctx = _ctx_for(Y, ctx)
    s = Solver(ctx, params, keep_blocks=keep_blocks)
    log = create_log(params)
    err = []

    def on_iter(_user, _solver, _done, _d):          # vbmf_b200_iter_callback: runs on this thread after every iteration
        try:
            s.download(params)
            update_log_(log, params)
            return 0
        except Exception as e:                       # never raise across the C ABI
            err.append(e)
            return 1
    cb = L_.ITER_CALLBACK(on_iter)
    it, d = C.c_int64(), C.c_double()
    try:
        s.upload(params)
        rc = L_.check(ctx.lib.vbmf_b200_solver_run_logged(s.h, int(niter), float(eps), flags, _NORMS[norm], cb, None, C.byref(it), C.byref(d)),
                      allow=(-2,))
        if err:
            raise err[0]
        _not_pd(rc, params)
        s.download(params, want_yhat=True)
    finally:
        s.close()
    it_total, d = it.value, d.value
    save_log(log, Y if Y is not None else np.zeros((0, 0)), {}, logdir, desc)
    return it_total, d, log
