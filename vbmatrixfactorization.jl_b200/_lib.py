"""ctypes binding of include/vbmf_b200.h (the C ABI a Julia `ccall` shim binds as well).  No torch types cross it."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libvbmf_b200.so")

c_i64 = C.c_int64
c_f64 = C.c_double
# data pointers travel as plain addresses (c_void_p): assigning an int is ~10x cheaper than building a typed ctypes pointer,
# which matters when thousands of small state structs are marshalled (batched vbls)
p_f64 = C.c_void_p
p_i64 = C.c_void_p

DENSE, SPARSE, DUAL, TRIAL = 0, 1, 2, 3
NORM_SPECTRAL, NORM_FROBENIUS = 0, 1
DIAG_VAR, FULL_COV, EST_CB, EST_PRIORS, EST_COVS, EST_VAR = 1, 2, 4, 8, 16, 32
(STEP_UPDATE_A, STEP_UPDATE_B, STEP_UPDATE_CA, STEP_UPDATE_CB, STEP_UPDATE_SIGMA, STEP_UPDATE_ALPHA00,
 STEP_UPDATE_ALPHA01, STEP_UPDATE_BETA00, STEP_UPDATE_BETA01, STEP_UPDATE_ALPHA02, STEP_UPDATE_BETA02) = range(11)


class DenseState(C.Structure):
    _fields_ = [("L", c_i64), ("M", c_i64), ("H", c_i64), ("H1", c_i64), ("n_labels", c_i64), ("labels", p_i64),
                ("AHat", p_f64), ("BHat", p_f64), ("SigmaA", p_f64), ("SigmaB", p_f64), ("CA", p_f64), ("CB", p_f64),
                ("invCA", p_f64), ("invCB", p_f64), ("sigma2", c_f64), ("YHat", p_f64)]


class SparseState(C.Structure):
    _fields_ = [("L", c_i64), ("M", c_i64), ("H", c_i64), ("MH", c_i64), ("H1", c_i64), ("n_labels", c_i64),
                ("labels", p_i64), ("AHat", p_f64), ("ATVecHat", p_f64), ("SigmaATVec_blocks", p_f64),
                ("diagSigmaATVec", p_f64), ("SigmaA", p_f64), ("BHat", p_f64), ("SigmaB", p_f64), ("CA", p_f64),
                ("alpha0", c_f64), ("beta0", c_f64), ("alpha", c_f64), ("beta", p_f64), ("CB", p_f64),
                ("gamma0", c_f64), ("delta0", c_f64), ("gamma", c_f64), ("delta", p_f64),
                ("sigmaHat", c_f64), ("eta0", c_f64), ("zeta0", c_f64), ("eta", c_f64), ("zeta", c_f64),
                ("sigmaVecHat", p_f64), ("etaVec", p_f64), ("zetaVec", p_f64), ("YHat", p_f64), ("trYTY", c_f64)]


class DualState(C.Structure):
    _fields_ = [("L", c_i64), ("M", c_i64), ("MH", c_i64), ("H", c_i64), ("H0", c_i64), ("H1", c_i64),
                ("AHat", p_f64), ("ATVecHat", p_f64), ("SigmaATVec_blocks", p_f64), ("diagSigmaATVec", p_f64),
                ("SigmaA", p_f64), ("A0Hat", p_f64), ("A1Hat", p_f64), ("BHat", p_f64), ("SigmaB", p_f64),
                ("CA", p_f64), ("alpha", p_f64), ("beta", p_f64), ("CA0", p_f64),
                ("alpha00", c_f64), ("beta00", c_f64), ("alpha0", c_f64), ("beta0", p_f64), ("CA1", p_f64),
                ("alpha01", c_f64), ("beta01", c_f64), ("alpha1", c_f64), ("beta1", p_f64), ("CB", p_f64),
                ("gamma0", c_f64), ("delta0", c_f64), ("gamma", c_f64), ("delta", p_f64),
                ("sigmaHat", c_f64), ("eta0", c_f64), ("zeta0", c_f64), ("eta", c_f64), ("zeta", c_f64),
                ("sigmaVecHat", p_f64), ("etaVec", p_f64), ("zetaVec", p_f64), ("YHat", p_f64), ("trYTY", c_f64)]


class TrialState(C.Structure):
    _fields_ = [("L", c_i64), ("M", c_i64), ("M0", c_i64), ("M1", c_i64), ("MH", c_i64), ("H", c_i64), ("H0", c_i64), ("H1", c_i64),
                ("AHat", p_f64), ("ATVecHat", p_f64), ("SigmaATVec_blocks", p_f64), ("diagSigmaATVec", p_f64), ("SigmaA", p_f64),
                ("A1Hat", p_f64), ("A2Hat", p_f64), ("A3Hat", p_f64), ("BHat", p_f64), ("SigmaB", p_f64),
                ("CA", p_f64), ("alpha", p_f64), ("beta", p_f64),
                ("CA1", p_f64), ("alpha01", c_f64), ("beta01", c_f64), ("alpha1", c_f64), ("beta1", p_f64),
                ("CA2", p_f64), ("alpha02", c_f64), ("beta02", c_f64), ("alpha2", c_f64), ("beta2", p_f64),
                ("CA3", p_f64), ("alpha03", c_f64), ("beta03", c_f64), ("alpha3", c_f64), ("beta3", p_f64),
                ("CB", p_f64), ("gamma0", c_f64), ("delta0", c_f64), ("gamma", c_f64), ("delta", p_f64),
                ("sigmaHat", c_f64), ("eta0", c_f64), ("zeta0", c_f64), ("eta", c_f64), ("zeta", c_f64),
                ("sigmaVecHat", p_f64), ("etaVec", p_f64), ("zetaVec", p_f64), ("YHat", p_f64), ("trYTY", c_f64)]


ITER_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, c_i64, c_f64)     # vbmf_b200_iter_callback

# every symbol include/vbmf_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "vbmf_b200_version": (C.c_int, []),
    "vbmf_b200_last_error": (C.c_char_p, []),
    "vbmf_b200_device_count": (C.c_int, []),
    "vbmf_b200_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "vbmf_b200_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "vbmf_b200_ctx_destroy": (C.c_int, [C.c_void_p]),
    "vbmf_b200_attach_Y": (C.c_int, [C.c_void_p, p_f64, c_i64, c_i64, c_i64, c_i64, c_i64]),
    "vbmf_b200_set_shape": (C.c_int, [C.c_void_p, c_i64, c_i64, c_i64, c_i64]),
    "vbmf_b200_synth_Y": (C.c_int, [C.c_void_p, c_i64, c_i64, c_i64, c_i64, C.c_int, c_f64, C.c_uint64]),
    "vbmf_b200_preprocess_Y": (C.c_int, [C.c_void_p, c_f64, p_i64, p_i64]),
    "vbmf_b200_download_Y": (C.c_int, [C.c_void_p, p_f64, c_i64]),
    "vbmf_b200_trYTY": (C.c_int, [C.c_void_p, p_f64]),
    "vbmf_b200_ctx_sync": (C.c_int, [C.c_void_p]),
    "vbmf_b200_launch_count": (c_i64, []),
    "vbmf_b200_plan_contractions": (C.c_int, [c_i64, c_i64, c_i64, C.c_int, p_i64]),
    "vbmf_b200_ctx_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "vbmf_b200_ctx_profile_read": (C.c_int, [C.c_void_p, p_f64, p_i64, p_f64, p_i64]),
    "vbmf_b200_ctx_profile_read_allreduce": (C.c_int, [C.c_void_p, p_f64, p_i64]),
    "vbmf_b200_ctx_peer_exchange": (C.c_int, [C.c_void_p]),
    "vbmf_b200_px_plan": (C.c_int, [C.c_int64, C.c_int, C.c_int, p_i64]),
    "vbmf_b200_ctx_profile_read_segments": (C.c_int, [C.c_void_p, p_f64, p_i64, C.c_int]),
    "vbmf_b200_gemm_YtB": (C.c_int, [C.c_void_p, p_f64, c_i64, p_f64]),
    "vbmf_b200_gemm_YA": (C.c_int, [C.c_void_p, p_f64, c_i64, p_f64]),
    "vbmf_b200_solver_create": (C.c_int, [C.c_void_p, C.c_int, c_i64, c_i64, c_i64, p_i64, C.c_int, C.POINTER(C.c_void_p)]),
    "vbmf_b200_solver_create_trial": (C.c_int, [C.c_void_p, c_i64, c_i64, c_i64, C.c_int, C.POINTER(C.c_void_p)]),
    "vbmf_b200_solver_destroy": (C.c_int, [C.c_void_p]),
    "vbmf_b200_dense_upload": (C.c_int, [C.c_void_p, C.POINTER(DenseState)]),
    "vbmf_b200_dense_download": (C.c_int, [C.c_void_p, C.POINTER(DenseState)]),
    "vbmf_b200_sparse_upload": (C.c_int, [C.c_void_p, C.POINTER(SparseState)]),
    "vbmf_b200_sparse_download": (C.c_int, [C.c_void_p, C.POINTER(SparseState)]),
    "vbmf_b200_dual_upload": (C.c_int, [C.c_void_p, C.POINTER(DualState)]),
    "vbmf_b200_dual_download": (C.c_int, [C.c_void_p, C.POINTER(DualState)]),
    "vbmf_b200_trial_upload": (C.c_int, [C.c_void_p, C.POINTER(TrialState)]),
    "vbmf_b200_trial_download": (C.c_int, [C.c_void_p, C.POINTER(TrialState)]),
    "vbmf_b200_solver_step": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "vbmf_b200_solver_run": (C.c_int, [C.c_void_p, c_i64, c_f64, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_solver_run_group": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, c_i64, c_f64, C.c_int, p_i64, p_f64, C.c_void_p]),
    "vbmf_b200_solver_run_logged": (C.c_int, [C.c_void_p, c_i64, c_f64, C.c_int, C.c_int, ITER_CALLBACK, C.c_void_p, p_i64, p_f64]),
    "vbmf_b200_solver_lower_bound": (C.c_int, [C.c_void_p, c_f64, C.c_int, p_f64]),
    "vbmf_b200_solver_yhat": (C.c_int, [C.c_void_p, p_f64, c_i64]),
    "vbmf_b200_batched_vbls": (C.c_int, [C.c_void_p, C.c_int, c_i64, C.POINTER(p_f64), C.POINTER(C.c_void_p), c_i64, C.c_int]),
    "vbmf_b200_batched_plan": (C.c_int, [C.c_int, c_i64, c_i64, C.c_int, C.c_int, c_i64, p_i64, C.c_void_p]),
    "vbmf_b200_batched_lower_bound": (C.c_int, [C.c_void_p, C.c_int, c_i64, C.POINTER(p_f64), C.POINTER(C.c_void_p), c_f64, C.c_int, p_f64]),
    "vbmf_b200_batched_residual_norm": (C.c_int, [C.c_void_p, C.c_int, c_i64, C.POINTER(p_f64), C.POINTER(C.c_void_p), C.c_int, p_f64]),
    "vbmf_b200_dense_run": (C.c_int, [C.c_void_p, C.POINTER(DenseState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_sparse_run": (C.c_int, [C.c_void_p, C.POINTER(SparseState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_dual_run": (C.c_int, [C.c_void_p, C.POINTER(DualState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_trial_run": (C.c_int, [C.c_void_p, C.POINTER(TrialState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    # several GPUs from one host process (csrc/multi.cu)
    "vbmf_b200_mctx_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "vbmf_b200_mctx_destroy": (C.c_int, [C.c_void_p]),
    "vbmf_b200_mctx_ndev": (C.c_int, [C.c_void_p]),
    "vbmf_b200_mctx_ctx": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "vbmf_b200_mctx_shard": (C.c_int, [C.c_void_p, C.c_int, p_i64, p_i64]),
    "vbmf_b200_mctx_attach_Y": (C.c_int, [C.c_void_p, p_f64, c_i64, c_i64, c_i64]),
    "vbmf_b200_mctx_synth_Y": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_int, c_f64, C.c_uint64]),
    "vbmf_b200_mctx_trYTY": (C.c_int, [C.c_void_p, p_f64]),
    "vbmf_b200_mctx_dense_run": (C.c_int, [C.c_void_p, C.POINTER(DenseState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_mctx_sparse_run": (C.c_int, [C.c_void_p, C.POINTER(SparseState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_mctx_dual_run": (C.c_int, [C.c_void_p, C.POINTER(DualState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_mctx_trial_run": (C.c_int, [C.c_void_p, C.POINTER(TrialState), c_i64, c_f64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, p_i64, p_f64]),
    "vbmf_b200_mctx_lower_bound": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, c_f64, C.c_int, p_f64]),
}

_lib = None


class VBMFError(RuntimeError):
    """Raised for every non-zero ABI return (the Julia shim turns the same condition into error(msg))."""


def load():
    """Load libvbmf_b200.so.  Fails loudly when it has not been built: there is no Python/CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VBMFError("%s is missing: run `python __graft_entry__.py` (build()) first; vbmf_b200 has no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, allow=()):
    if rc != 0 and rc not in allow:
        msg = load().vbmf_b200_last_error()
        raise VBMFError((msg or b"unknown error").decode("utf-8", "replace"))
    return rc
