# VBMatrixFactorizationB200.jl -- thin `ccall` shim that routes VBMatrixFactorization.jl's VB update loop to libvbmf_b200.so.
#
# Drop-in for the hot path only: `vbmf!`, `vbmf_sparse!`, `vbmf_dual!` (and the non-mutating `vbmf`, `vbmf_sparse`, `vbmf_dual`),
# `lowerBound`, `lowerBoundTrimmed` keep their reference signatures (src/vbmf.jl:175,238; src/vbmf_sparse.jl:344,418,435,478;
# src/vbmf_dual.jl:455,538,556,606).  Everything else (init = Julia RNG, preprocessing, logging, MIL scripts) stays in the
# reference package.  Written in the reference's dialect (Julia 0.5: `type`, `immutable`, `Ptr{Void}`); on Julia >= 1.0
# replace `immutable` by `struct`, `Void` by `Cvoid`.  NOT EXECUTED in the build container (no Julia toolchain there): the same
# ABI is exercised by the ctypes binding (vbmatrixfactorization.jl_b200/_lib.py) in tests/.
#
# Usage:  include("VBMatrixFactorizationB200.jl"); using VBMatrixFactorizationB200
#         vbmf!(Y, params, 100, est_covs = true, est_var = true)         # the reference's call, now on GPU 0
#         b200_default_context!(b200_context(0:7))                       # ... or on all eight GPUs of the box, same call
#         ctx = b200_context(1); vbmf!(ctx, Y, params, 100)              # explicit context; vbmf!(ctx, nothing, ...) = Y resident
module VBMatrixFactorizationB200

using VBMatrixFactorization
import VBMatrixFactorization: vbmf_parameters, vbmf_sparse_parameters, vbmf_dual_parameters, vbmf_trial_parameters
# extended (and, for the reference's own signatures, replaced) by the methods below
import VBMatrixFactorization: vbmf!, vbmf, vbmf_sparse!, vbmf_sparse, vbmf_dual!, vbmf_dual, vbmf_trial!, vbmf_trial,
                              lowerBound, lowerBoundTrimmed

export b200_context, b200_close, b200_peer_exchange, b200_default_context!, vbmf!, vbmf, vbmf_sparse!, vbmf_sparse, vbmf_dual!, vbmf_dual, vbmf_trial!, vbmf_trial,
       lowerBound, lowerBoundTrimmed, vbls_batched!, lowerBound_batched, lowerBoundTrimmed_batched, preprocess

const LIB = get(ENV, "VBMF_B200_LIB", "libvbmf_b200.so")

# ---- mirrors of the C structs in include/vbmf_b200.h (all fields 8 bytes, same order) -------------------------------------
immutable DenseState        # vbmf_b200_dense_state  <->  vbmf_parameters (src/vbmf.jl:22-40)
    L::Int64; M::Int64; H::Int64; H1::Int64
    n_labels::Int64; labels::Ptr{Int64}
    AHat::Ptr{Float64}; BHat::Ptr{Float64}; SigmaA::Ptr{Float64}; SigmaB::Ptr{Float64}
    CA::Ptr{Float64}; CB::Ptr{Float64}; invCA::Ptr{Float64}; invCB::Ptr{Float64}
    sigma2::Float64
    YHat::Ptr{Float64}
end

immutable SparseState       # vbmf_b200_sparse_state <->  vbmf_sparse_parameters (src/vbmf_sparse.jl:47-90)
    L::Int64; M::Int64; H::Int64; MH::Int64; H1::Int64
    n_labels::Int64; labels::Ptr{Int64}
    AHat::Ptr{Float64}; ATVecHat::Ptr{Float64}; SigmaATVec_blocks::Ptr{Float64}; diagSigmaATVec::Ptr{Float64}
    SigmaA::Ptr{Float64}; BHat::Ptr{Float64}; SigmaB::Ptr{Float64}; CA::Ptr{Float64}
    alpha0::Float64; beta0::Float64; alpha::Float64; beta::Ptr{Float64}
    CB::Ptr{Float64}; gamma0::Float64; delta0::Float64; gamma::Float64; delta::Ptr{Float64}
    sigmaHat::Float64; eta0::Float64; zeta0::Float64; eta::Float64; zeta::Float64
    sigmaVecHat::Ptr{Float64}; etaVec::Ptr{Float64}; zetaVec::Ptr{Float64}
    YHat::Ptr{Float64}; trYTY::Float64
end

immutable DualState         # vbmf_b200_dual_state   <->  vbmf_dual_parameters (src/vbmf_dual.jl:59-112)
    L::Int64; M::Int64; MH::Int64; H::Int64; H0::Int64; H1::Int64
    AHat::Ptr{Float64}; ATVecHat::Ptr{Float64}; SigmaATVec_blocks::Ptr{Float64}; diagSigmaATVec::Ptr{Float64}
    SigmaA::Ptr{Float64}; A0Hat::Ptr{Float64}; A1Hat::Ptr{Float64}; BHat::Ptr{Float64}; SigmaB::Ptr{Float64}
    CA::Ptr{Float64}; alpha::Ptr{Float64}; beta::Ptr{Float64}; CA0::Ptr{Float64}
    alpha00::Float64; beta00::Float64; alpha0::Float64; beta0::Ptr{Float64}; CA1::Ptr{Float64}
    alpha01::Float64; beta01::Float64; alpha1::Float64; beta1::Ptr{Float64}; CB::Ptr{Float64}
    gamma0::Float64; delta0::Float64; gamma::Float64; delta::Ptr{Float64}
    sigmaHat::Float64; eta0::Float64; zeta0::Float64; eta::Float64; zeta::Float64
    sigmaVecHat::Ptr{Float64}; etaVec::Ptr{Float64}; zetaVec::Ptr{Float64}
    YHat::Ptr{Float64}; trYTY::Float64
end

immutable TrialState        # vbmf_b200_trial_state  <->  vbmf_trial_parameters (src/vbmf_trial.jl:68-129)
    L::Int64; M::Int64; M0::Int64; M1::Int64; MH::Int64; H::Int64; H0::Int64; H1::Int64
    AHat::Ptr{Float64}; ATVecHat::Ptr{Float64}; SigmaATVec_blocks::Ptr{Float64}; diagSigmaATVec::Ptr{Float64}; SigmaA::Ptr{Float64}
    A1Hat::Ptr{Float64}; A2Hat::Ptr{Float64}; A3Hat::Ptr{Float64}; BHat::Ptr{Float64}; SigmaB::Ptr{Float64}
    CA::Ptr{Float64}; alpha::Ptr{Float64}; beta::Ptr{Float64}
    CA1::Ptr{Float64}; alpha01::Float64; beta01::Float64; alpha1::Float64; beta1::Ptr{Float64}
    CA2::Ptr{Float64}; alpha02::Float64; beta02::Float64; alpha2::Float64; beta2::Ptr{Float64}
    CA3::Ptr{Float64}; alpha03::Float64; beta03::Float64; alpha3::Float64; beta3::Ptr{Float64}
    CB::Ptr{Float64}; gamma0::Float64; delta0::Float64; gamma::Float64; delta::Ptr{Float64}
    sigmaHat::Float64; eta0::Float64; zeta0::Float64; eta::Float64; zeta::Float64
    sigmaVecHat::Ptr{Float64}; etaVec::Ptr{Float64}; zetaVec::Ptr{Float64}
    YHat::Ptr{Float64}; trYTY::Float64
end

# One GPU (vbmf_b200_ctx) or several GPUs driven from this one Julia process (vbmf_b200_mctx: the library splits the columns
# of Y over the devices, one host thread per device, NCCL all-reduce inside the loop).
type B200Context
    handle::Ptr{Void}
    multi::Bool
    ndev::Int
end

# 0 ok; -2 = a posterior precision matrix was not positive definite (NaN written, loop ended): the reference's LU `inv` would
# return garbage or throw SingularException there -- surfaced as a warning with the library's message; anything else: error
function check(rc)
    rc == 0 && return true
    msg = unsafe_string(ccall((:vbmf_b200_last_error, LIB), Cstring, ()))
    rc == -2 ? warn("vbmf_b200: ", msg) : error(msg)
    return true
end

function b200_context(device::Int = 0)
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:vbmf_b200_ctx_create, LIB), Cint, (Cint, Cint, Cint, Ptr{Void}, Ptr{Void}, Ptr{Ptr{Void}}),
                device, 0, 1, C_NULL, C_NULL, h))
    return B200Context(h[], false, 1)
end
# b200_context(0:7): all eight GPUs of the box from this process
function b200_context(devices::AbstractVector)
    devs = Cint[d for d in devices]
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:vbmf_b200_mctx_create, LIB), Cint, (Cint, Ptr{Cint}, Ptr{Ptr{Void}}), length(devs), devs, h))
    return B200Context(h[], true, length(devs))
end
# Several GPUs: true when the per-iteration exchange of updateB! runs through peer-mapped memory over NVLink (the library's own
# kernels; world 2..8 on one node, H <= 64, decided when the first solver is created) instead of the NCCL all-reduce.
function b200_peer_exchange(ctx::B200Context)
    if !ctx.multi
        return ccall((:vbmf_b200_ctx_peer_exchange, LIB), Cint, (Ptr{Void},), ctx.handle) != 0
    end
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:vbmf_b200_mctx_ctx, LIB), Cint, (Ptr{Void}, Cint, Ptr{Ptr{Void}}), ctx.handle, 0, h))
    return ccall((:vbmf_b200_ctx_peer_exchange, LIB), Cint, (Ptr{Void},), h[]) != 0
end
b200_close(ctx::B200Context) = ctx.multi ? ccall((:vbmf_b200_mctx_destroy, LIB), Cint, (Ptr{Void},), ctx.handle) :
                                           ccall((:vbmf_b200_ctx_destroy, LIB), Cint, (Ptr{Void},), ctx.handle)

# The methods with the reference's exact signatures (no ctx argument) use this context; created on first use on device 0,
# or set it to a multi-GPU context: b200_default_context!(b200_context(0:7)).
const DEFAULT_CTX = Ref{Any}(nothing)
b200_default_context!(ctx::B200Context) = (DEFAULT_CTX[] = ctx)
default_context() = (DEFAULT_CTX[] === nothing && (DEFAULT_CTX[] = b200_context(0)); DEFAULT_CTX[]::B200Context)

# Y is uploaded on every call that receives it: the library never guesses that a host array is unchanged (an in-place edit is
# invisible to any identity check).  To keep Y resident across calls, attach it once and pass `nothing` for Y afterwards.
function attach!(ctx::B200Context, Y::Array{Float64,2})
    L, M = size(Y)
    if ctx.multi
        check(ccall((:vbmf_b200_mctx_attach_Y, LIB), Cint, (Ptr{Void}, Ptr{Float64}, Int64, Int64, Int64), ctx.handle, Y, L, M, L))
    else
        check(ccall((:vbmf_b200_attach_Y, LIB), Cint, (Ptr{Void}, Ptr{Float64}, Int64, Int64, Int64, Int64, Int64),
                    ctx.handle, Y, L, M, L, M, 0))
    end
end
attach!(ctx::B200Context, Y::Void) = nothing          # Y already resident

const NORM = Dict(:spectral => 0, :frobenius => 1)   # :spectral = Julia 0.5 norm(::Matrix), what src/util.jl:28 computes
# updateYHat! runs after the loop in the reference (src/vbmf.jl:216); YHat is L x M (32 GB at 20000 x 200000), so it is only
# allocated when asked for (yhat = true, the reference's behaviour, is the default; pass yhat = false at scale)
yhat_buffer(p, yhat::Bool) = yhat ? Array{Float64}(p.L, p.M) : Array{Float64}(0, 0)
yhat_ptr(p, yhat::Bool) = yhat ? pointer(p.YHat) : convert(Ptr{Float64}, C_NULL)
sym(ctx::B200Context, single::Symbol, multi::Symbol) = ctx.multi ? multi : single

# logdir != "": the reference's create_log / update_log! / save_log (src/data_manip.jl:6-66, JLD on disk) around one device
# iteration at a time -- the log format on disk is the reference's own, written by the reference's own functions
function logged(run1!, Y, p, niter::Int, eps::Float64, logdir::String, desc::String)
    log = VBMatrixFactorization.create_log(p)
    priors = Dict{Any,Any}()
    d = eps + 1.0; i = 1
    while i <= niter && d > eps
        d = run1!()
        VBMatrixFactorization.update_log!(log, p)
        i += 1
    end
    VBMatrixFactorization.save_log(log, Y, priors, logdir, desc = desc)
    return d, i - 1
end

# ---- vbmf! (src/vbmf.jl:175) ----------------------------------------------------------------------------------------------
function dense_call!(ctx::B200Context, p::vbmf_parameters, niter::Int, eps, est_covs, est_var, norm, yhat::Bool)
    p.YHat = yhat_buffer(p, yhat)
    st = Ref(DenseState(p.L, p.M, p.H, p.H1, length(p.labels), pointer(p.labels), pointer(p.AHat), pointer(p.BHat),
                        pointer(p.SigmaA), pointer(p.SigmaB), pointer(p.CA), pointer(p.CB), pointer(p.invCA), pointer(p.invCB),
                        p.sigma2, yhat_ptr(p, yhat)))
    iters = Ref{Int64}(0); d = Ref{Float64}(0.0)
    if ctx.multi
        check(ccall((:vbmf_b200_mctx_dense_run, LIB), Cint,
                    (Ptr{Void}, Ref{DenseState}, Int64, Float64, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, est_covs, est_var, NORM[norm], iters, d))
    else
        check(ccall((:vbmf_b200_dense_run, LIB), Cint,
                    (Ptr{Void}, Ref{DenseState}, Int64, Float64, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, est_covs, est_var, NORM[norm], iters, d))
    end
    p.sigma2 = st[].sigma2
    return iters[], d[]
end
function vbmf!(ctx::B200Context, Y, p::vbmf_parameters, niter::Int; eps::Float64 = 1e-6, est_covs::Bool = false,
               est_var::Bool = false, logdir = "", desc = "", verb = false, norm = :spectral, yhat::Bool = true)
    attach!(ctx, Y)
    if logdir != ""
        d, iters = logged(() -> dense_call!(ctx, p, 1, eps, est_covs, est_var, norm, false)[2], Y, p, niter, eps, logdir, desc)
        yhat && dense_call!(ctx, p, 0, eps, est_covs, est_var, norm, true)          # updateYHat! after the loop
    else
        iters, d = dense_call!(ctx, p, niter, eps, est_covs, est_var, norm, yhat)
    end
    verb && print("Factorization finished after ", iters, " iterations, eps = ", d, "\n")
    return p
end
vbmf(ctx::B200Context, Y, p_in::vbmf_parameters, niter::Int; kw...) = vbmf!(ctx, Y, deepcopy(p_in), niter; kw...)
# the reference's own signatures (src/vbmf.jl:175,238): these REPLACE the CPU methods of the loaded reference package
vbmf!(Y::Array{Float64,2}, p::vbmf_parameters, niter::Int; kw...) = vbmf!(default_context(), Y, p, niter; kw...)
vbmf(Y::Array{Float64,2}, p_in::vbmf_parameters, niter::Int; kw...) = vbmf(default_context(), Y, p_in, niter; kw...)

# ---- vbmf_sparse! (src/vbmf_sparse.jl:344) ----------------------------------------------------------------------------------
function sparse_state(p::vbmf_sparse_parameters, blocks::Ptr{Float64}, yhat::Bool = true)
    SparseState(p.L, p.M, p.H, p.MH, p.H1, length(p.labels), pointer(p.labels), pointer(p.AHat), pointer(p.ATVecHat), blocks,
                pointer(p.diagSigmaATVec), pointer(p.SigmaA), pointer(p.BHat), pointer(p.SigmaB), pointer(p.CA),
                p.alpha0, p.beta0, p.alpha, pointer(p.beta), pointer(p.CB), p.gamma0, p.delta0, p.gamma, pointer(p.delta),
                p.sigmaHat, p.eta0, p.zeta0, p.eta, p.zeta, pointer(p.sigmaVecHat), pointer(p.etaVec), pointer(p.zetaVec),
                yhat_ptr(p, yhat), p.trYTY)
end
function sparse_call!(ctx::B200Context, p::vbmf_sparse_parameters, niter::Int, eps, diag_var, full_cov, est_cb, norm, yhat::Bool)
    p.YHat = yhat_buffer(p, yhat)
    # the (MH)x(MH) SigmaATVec / invSigmaATVec of the reference are never materialised; ask for the M diagonal blocks with
    # blocks = Array{Float64}(p.H, p.H, p.M) and pass pointer(blocks) instead of C_NULL when they are needed.
    st = Ref(sparse_state(p, convert(Ptr{Float64}, C_NULL), yhat))
    iters = Ref{Int64}(0); d = Ref{Float64}(0.0)
    if ctx.multi
        check(ccall((:vbmf_b200_mctx_sparse_run, LIB), Cint,
                    (Ptr{Void}, Ref{SparseState}, Int64, Float64, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_cb, NORM[norm], iters, d))
    else
        check(ccall((:vbmf_b200_sparse_run, LIB), Cint,
                    (Ptr{Void}, Ref{SparseState}, Int64, Float64, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_cb, NORM[norm], iters, d))
    end
    p.sigmaHat = st[].sigmaHat; p.zeta = st[].zeta
    return iters[], d[]
end
function vbmf_sparse!(ctx::B200Context, Y, p::vbmf_sparse_parameters, niter::Int; eps::Float64 = 1e-6, diag_var::Bool = false,
                      full_cov::Bool = false, logdir = "", desc = "", verb = false, est_cb::Bool = true, norm = :spectral,
                      yhat::Bool = true)
    attach!(ctx, Y)
    if logdir != ""
        d, iters = logged(() -> sparse_call!(ctx, p, 1, eps, diag_var, full_cov, est_cb, norm, false)[2], Y, p, niter, eps, logdir, desc)
        yhat && sparse_call!(ctx, p, 0, eps, diag_var, full_cov, est_cb, norm, true)
    else
        iters, d = sparse_call!(ctx, p, niter, eps, diag_var, full_cov, est_cb, norm, yhat)
    end
    verb && print("Factorization finished after ", iters, " iterations, eps = ", d, "\n")
    return d
end
function vbmf_sparse(ctx::B200Context, Y, p_in::vbmf_sparse_parameters, niter::Int; kw...)
    p = deepcopy(p_in)
    d = vbmf_sparse!(ctx, Y, p, niter; kw...)
    return p, d
end
vbmf_sparse!(Y::Array{Float64,2}, p::vbmf_sparse_parameters, niter::Int; kw...) = vbmf_sparse!(default_context(), Y, p, niter; kw...)
vbmf_sparse(Y::Array{Float64,2}, p_in::vbmf_sparse_parameters, niter::Int; kw...) = vbmf_sparse(default_context(), Y, p_in, niter; kw...)

# ---- vbmf_dual! (src/vbmf_dual.jl:455) ----------------------------------------------------------------------------------------
function dual_state(p::vbmf_dual_parameters, yhat::Bool = true)
    DualState(p.L, p.M, p.MH, p.H, p.H0, p.H1, pointer(p.AHat), pointer(p.ATVecHat), convert(Ptr{Float64}, C_NULL),
              pointer(p.diagSigmaATVec), pointer(p.SigmaA), pointer(p.A0Hat), pointer(p.A1Hat), pointer(p.BHat), pointer(p.SigmaB),
              pointer(p.CA), pointer(p.alpha), pointer(p.beta), pointer(p.CA0), p.alpha00, p.beta00, p.alpha0, pointer(p.beta0),
              pointer(p.CA1), p.alpha01, p.beta01, p.alpha1, pointer(p.beta1), pointer(p.CB), p.gamma0, p.delta0, p.gamma,
              pointer(p.delta), p.sigmaHat, p.eta0, p.zeta0, p.eta, p.zeta, pointer(p.sigmaVecHat), pointer(p.etaVec),
              pointer(p.zetaVec), yhat_ptr(p, yhat), p.trYTY)
end
function dual_call!(ctx::B200Context, p::vbmf_dual_parameters, niter::Int, eps, diag_var, full_cov, est_priors, est_cb, norm, yhat::Bool)
    p.YHat = yhat_buffer(p, yhat)
    st = Ref(dual_state(p, yhat))
    iters = Ref{Int64}(0); d = Ref{Float64}(0.0)
    if ctx.multi
        check(ccall((:vbmf_b200_mctx_dual_run, LIB), Cint,
                    (Ptr{Void}, Ref{DualState}, Int64, Float64, Cint, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_priors, est_cb, NORM[norm], iters, d))
    else
        check(ccall((:vbmf_b200_dual_run, LIB), Cint,
                    (Ptr{Void}, Ref{DualState}, Int64, Float64, Cint, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_priors, est_cb, NORM[norm], iters, d))
    end
    s = st[]
    p.sigmaHat = s.sigmaHat; p.zeta = s.zeta
    p.alpha00 = s.alpha00; p.beta00 = s.beta00; p.alpha01 = s.alpha01; p.beta01 = s.beta01
    p.alpha0 = s.alpha0; p.alpha1 = s.alpha1
    return iters[], d[]
end
function vbmf_dual!(ctx::B200Context, Y, p::vbmf_dual_parameters, niter::Int; eps::Float64 = 1e-6, diag_var::Bool = false,
                    full_cov::Bool = false, logdir = "", desc = "", verb = false, est_priors = true, est_cb::Bool = true,
                    norm = :spectral, yhat::Bool = true)
    attach!(ctx, Y)
    if logdir != ""
        d, iters = logged(() -> dual_call!(ctx, p, 1, eps, diag_var, full_cov, est_priors, est_cb, norm, false)[2], Y, p, niter, eps, logdir, desc)
        yhat && dual_call!(ctx, p, 0, eps, diag_var, full_cov, est_priors, est_cb, norm, true)
    else
        iters, d = dual_call!(ctx, p, niter, eps, diag_var, full_cov, est_priors, est_cb, norm, yhat)
    end
    verb && print("Factorization finished after ", iters, " iterations, eps = ", d, "\n")
    return d
end
function vbmf_dual(ctx::B200Context, Y, p_in::vbmf_dual_parameters, niter::Int; kw...)
    p = deepcopy(p_in)
    d = vbmf_dual!(ctx, Y, p, niter; kw...)
    return p, d
end
vbmf_dual!(Y::Array{Float64,2}, p::vbmf_dual_parameters, niter::Int; kw...) = vbmf_dual!(default_context(), Y, p, niter; kw...)
vbmf_dual(Y::Array{Float64,2}, p_in::vbmf_dual_parameters, niter::Int; kw...) = vbmf_dual(default_context(), Y, p_in, niter; kw...)

# ---- vbmf_trial! (src/vbmf_trial.jl:528) -----------------------------------------------------------------------------------------
function trial_state(p::vbmf_trial_parameters, yhat::Bool = true)
    TrialState(p.L, p.M, p.M0, p.M1, p.MH, p.H, p.H0, p.H1, pointer(p.AHat), pointer(p.ATVecHat), convert(Ptr{Float64}, C_NULL),
               pointer(p.diagSigmaATVec), pointer(p.SigmaA), pointer(p.A1Hat), pointer(p.A2Hat), pointer(p.A3Hat), pointer(p.BHat),
               pointer(p.SigmaB), pointer(p.CA), pointer(p.alpha), pointer(p.beta),
               pointer(p.CA1), p.alpha01, p.beta01, p.alpha1, pointer(p.beta1), pointer(p.CA2), p.alpha02, p.beta02, p.alpha2, pointer(p.beta2),
               pointer(p.CA3), p.alpha03, p.beta03, p.alpha3, pointer(p.beta3), pointer(p.CB), p.gamma0, p.delta0, p.gamma, pointer(p.delta),
               p.sigmaHat, p.eta0, p.zeta0, p.eta, p.zeta, pointer(p.sigmaVecHat), pointer(p.etaVec), pointer(p.zetaVec), yhat_ptr(p, yhat), p.trYTY)
end
function vbmf_trial!(ctx::B200Context, Y, p::vbmf_trial_parameters, niter::Int; eps::Float64 = 1e-6, diag_var::Bool = false,
                     full_cov::Bool = false, verb = false, est_priors = true, est_cb::Bool = true, norm = :spectral, yhat::Bool = true)
    attach!(ctx, Y)
    p.YHat = yhat_buffer(p, yhat)
    st = Ref(trial_state(p, yhat))
    iters = Ref{Int64}(0); d = Ref{Float64}(0.0)
    if ctx.multi
        check(ccall((:vbmf_b200_mctx_trial_run, LIB), Cint,
                    (Ptr{Void}, Ref{TrialState}, Int64, Float64, Cint, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_priors, est_cb, NORM[norm], iters, d))
    else
        check(ccall((:vbmf_b200_trial_run, LIB), Cint,
                    (Ptr{Void}, Ref{TrialState}, Int64, Float64, Cint, Cint, Cint, Cint, Cint, Ref{Int64}, Ref{Float64}),
                    ctx.handle, st, niter, eps, diag_var, full_cov, est_priors, est_cb, NORM[norm], iters, d))
    end
    s = st[]
    p.sigmaHat = s.sigmaHat; p.zeta = s.zeta
    p.alpha01 = s.alpha01; p.beta01 = s.beta01; p.alpha02 = s.alpha02; p.beta02 = s.beta02; p.alpha03 = s.alpha03; p.beta03 = s.beta03
    p.alpha1 = s.alpha1; p.alpha2 = s.alpha2; p.alpha3 = s.alpha3
    verb && print("Factorization finished after ", iters[], " iterations, eps = ", d[], "\n")
    return d[]
end
function vbmf_trial(ctx::B200Context, Y, p_in::vbmf_trial_parameters, niter::Int; kw...)
    p = deepcopy(p_in)
    d = vbmf_trial!(ctx, Y, p, niter; kw...)
    return p, d
end
vbmf_trial!(Y::Array{Float64,2}, p::vbmf_trial_parameters, niter::Int; kw...) = vbmf_trial!(default_context(), Y, p, niter; kw...)
vbmf_trial(Y::Array{Float64,2}, p_in::vbmf_trial_parameters, niter::Int; kw...) = vbmf_trial(default_context(), Y, p_in, niter; kw...)

# ---- vbls! for many bags in one call (examples/mil_util.jl:179-203, 504-511) ----------------------------------------------------
# Ys[k] is the L x M_k matrix of problem k, ps[k] its parameters (all of one type, with the same L, H, H0); one method per
# branch of vbls! (:182-197).  kind: 0 dense, 1 sparse, 2 dual, 3 trial (include/vbmf_b200.h).  Bags of any size: those
# too large for one CTA's shared memory run in the wide kernel (one thread-block cluster per bag) within the same call.
function batched_call(ctx::B200Context, kind::Int, Ys::Vector{Array{Float64,2}}, sts::Vector, niter::Int, flags::Int)
    yptr = Ptr{Float64}[pointer(Y) for Y in Ys]
    sptr = Ptr{Void}[convert(Ptr{Void}, Base.unsafe_convert(Ptr{eltype(r)}, r)) for r in sts]
    check(ccall((:vbmf_b200_batched_vbls, LIB), Cint, (Ptr{Void}, Cint, Int64, Ptr{Ptr{Float64}}, Ptr{Ptr{Void}}, Int64, Cint),
                ctx.handle, kind, length(sts), yptr, sptr, niter, flags))
end
function vbls_batched!(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_dual_parameters}, niter::Int; full_cov::Bool = false)
    for p in ps; p.YHat = Array{Float64}(p.L, p.M); end
    sts = [Ref(dual_state(p)) for p in ps]
    batched_call(ctx, 2, Ys, sts, niter, full_cov ? 2 : 0)
    for (p, r) in zip(ps, sts)
        p.sigmaHat = r[].sigmaHat; p.zeta = r[].zeta; p.alpha0 = r[].alpha0; p.alpha1 = r[].alpha1
    end
    return [p.AHat for p in ps]
end
function vbls_batched!(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_sparse_parameters}, niter::Int; full_cov::Bool = false)
    for p in ps; p.YHat = Array{Float64}(p.L, p.M); end
    sts = [Ref(sparse_state(p, convert(Ptr{Float64}, C_NULL))) for p in ps]
    batched_call(ctx, 1, Ys, sts, niter, full_cov ? 2 : 0)
    for (p, r) in zip(ps, sts)
        p.sigmaHat = r[].sigmaHat; p.zeta = r[].zeta
    end
    return [p.AHat for p in ps]
end
function vbls_batched!(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_trial_parameters}, niter::Int; full_cov::Bool = false)
    for p in ps; p.YHat = Array{Float64}(p.L, p.M); end
    sts = [Ref(trial_state(p)) for p in ps]
    batched_call(ctx, 3, Ys, sts, niter, full_cov ? 2 : 0)
    for (p, r) in zip(ps, sts)
        p.sigmaHat = r[].sigmaHat; p.zeta = r[].zeta; p.alpha1 = r[].alpha1; p.alpha2 = r[].alpha2; p.alpha3 = r[].alpha3
    end
    return [p.AHat for p in ps]
end
function vbls_batched!(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_parameters}, niter::Int)
    for p in ps; p.YHat = Array{Float64}(p.L, p.M); end
    sts = [Ref(DenseState(p.L, p.M, p.H, p.H1, length(p.labels), pointer(p.labels), pointer(p.AHat), pointer(p.BHat),
                          pointer(p.SigmaA), pointer(p.SigmaB), pointer(p.CA), pointer(p.CB), pointer(p.invCA), pointer(p.invCB),
                          p.sigma2, pointer(p.YHat))) for p in ps]
    batched_call(ctx, 0, Ys, sts, niter, 0)
    for (p, r) in zip(ps, sts); p.sigma2 = r[].sigma2; end
    return [p.AHat for p in ps]
end

# ---- lowerBound / lowerBoundTrimmed for many bags in one call (src/vbmf_sparse.jl:435-489, src/vbmf_dual.jl:556-617,
# src/vbmf_trial.jl:630-697): the ELBO of every (bag, class model) pair, e.g. after vbls_batched!.  Same grouping rules as
# vbls_batched! (one type, one L, H and H0; H <= 64); single-device contexts; needs no attached Y.  Returns a Vector{Float64}.
function batched_lb_call(ctx::B200Context, kind::Int, Ys::Vector{Array{Float64,2}}, sts::Vector, trim::Float64, trimmed::Bool)
    ctx.multi && error("the batched lowerBound runs on one device: use a single-device context")
    yptr = Ptr{Float64}[pointer(Y) for Y in Ys]
    sptr = Ptr{Void}[convert(Ptr{Void}, Base.unsafe_convert(Ptr{eltype(r)}, r)) for r in sts]
    out = Array{Float64}(length(sts))
    check(ccall((:vbmf_b200_batched_lower_bound, LIB), Cint,
                (Ptr{Void}, Cint, Int64, Ptr{Ptr{Float64}}, Ptr{Ptr{Void}}, Float64, Cint, Ptr{Float64}),
                ctx.handle, kind, length(sts), yptr, sptr, trim, trimmed, out))
    return out
end
function batched_lower_bound(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_sparse_parameters}, trim::Float64, trimmed::Bool)
    for p in ps; isdefined(p, :YHat) || (p.YHat = Array{Float64}(0, 0)); end
    batched_lb_call(ctx, 1, Ys, [Ref(sparse_state(p, convert(Ptr{Float64}, C_NULL), false)) for p in ps], trim, trimmed)
end
function batched_lower_bound(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_dual_parameters}, trim::Float64, trimmed::Bool)
    for p in ps; isdefined(p, :YHat) || (p.YHat = Array{Float64}(0, 0)); end
    batched_lb_call(ctx, 2, Ys, [Ref(dual_state(p, false)) for p in ps], trim, trimmed)
end
function batched_lower_bound(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_trial_parameters}, trim::Float64, trimmed::Bool)
    for p in ps; isdefined(p, :YHat) || (p.YHat = Array{Float64}(0, 0)); end
    batched_lb_call(ctx, 3, Ys, [Ref(trial_state(p, false)) for p in ps], trim, trimmed)
end
batched_lower_bound(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector{vbmf_parameters}, trim::Float64, trimmed::Bool) =
    error("the dense solver has no lowerBound (the reference defines none)")
lowerBound_batched(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector) = batched_lower_bound(ctx, Ys, ps, 0.0, false)
lowerBoundTrimmed_batched(ctx::B200Context, Ys::Vector{Array{Float64,2}}, ps::Vector, trim = 1e-1) =
    batched_lower_bound(ctx, Ys, ps, Float64(trim), true)

# ---- preprocess(Y, lambda) (src/util.jl:73-87) on the device; the processed matrix stays resident (pass `nothing` for Y to
# the solvers to run on it without another upload); single-device contexts
function preprocess(ctx::B200Context, Y::Array{Float64,2}, lambda::Float64; verb = false)
    ctx.multi && error("preprocess runs on a single-device context")
    attach!(ctx, Y)
    L, M = size(Y)
    Lnew = Ref{Int64}(0); rows = Array{Int64}(L)
    check(ccall((:vbmf_b200_preprocess_Y, LIB), Cint, (Ptr{Void}, Float64, Ref{Int64}, Ptr{Int64}), ctx.handle, lambda, Lnew, rows))
    verb && println("Original problem size: $L rows, $(L - Lnew[]) rows not relevant and are not used.")
    out = Array{Float64}(Lnew[], M)
    check(ccall((:vbmf_b200_download_Y, LIB), Cint, (Ptr{Void}, Ptr{Float64}, Int64), ctx.handle, out, Lnew[]))
    return out
end

# ---- lowerBound / lowerBoundTrimmed (src/vbmf_sparse.jl:435,478; src/vbmf_dual.jl:556,606) and the step functions -------------
# go through the resident-solver entry points: solver_create -> *_upload -> solver_lower_bound / solver_step -> *_download.
function with_solver(f, ctx::B200Context, kind::Int, H::Int, split::Int, labels::Vector{Int64})
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:vbmf_b200_solver_create, LIB), Cint, (Ptr{Void}, Cint, Int64, Int64, Int64, Ptr{Int64}, Cint, Ptr{Ptr{Void}}),
                ctx.handle, kind, H, split, length(labels), labels, 0, h))
    try
        return f(h[])
    finally
        ccall((:vbmf_b200_solver_destroy, LIB), Cint, (Ptr{Void},), h[])
    end
end
function lower_bound(ctx::B200Context, Y, p::vbmf_sparse_parameters, trim::Float64, trimmed::Bool)
    isdefined(p, :YHat) || (p.YHat = Array{Float64}(0, 0))
    ctx.multi && return multi_lower_bound(ctx, Y, 1, Ref(sparse_state(p, convert(Ptr{Float64}, C_NULL), false)), trim, trimmed)
    attach!(ctx, Y)
    with_solver(ctx, 1, p.H, p.H1, p.labels) do s
        st = Ref(sparse_state(p, convert(Ptr{Float64}, C_NULL), false))
        check(ccall((:vbmf_b200_sparse_upload, LIB), Cint, (Ptr{Void}, Ref{SparseState}), s, st))
        out = Ref{Float64}(0.0)
        check(ccall((:vbmf_b200_solver_lower_bound, LIB), Cint, (Ptr{Void}, Float64, Cint, Ref{Float64}), s, trim, trimmed, out))
        out[]
    end
end
function lower_bound(ctx::B200Context, Y, p::vbmf_dual_parameters, trim::Float64, trimmed::Bool)
    isdefined(p, :YHat) || (p.YHat = Array{Float64}(0, 0))
    ctx.multi && return multi_lower_bound(ctx, Y, 2, Ref(dual_state(p, false)), trim, trimmed)
    attach!(ctx, Y)
    with_solver(ctx, 2, p.H, p.H0, Int64[]) do s
        st = Ref(dual_state(p, false))
        check(ccall((:vbmf_b200_dual_upload, LIB), Cint, (Ptr{Void}, Ref{DualState}), s, st))
        out = Ref{Float64}(0.0)
        check(ccall((:vbmf_b200_solver_lower_bound, LIB), Cint, (Ptr{Void}, Float64, Cint, Ref{Float64}), s, trim, trimmed, out))
        out[]
    end
end
function multi_lower_bound(ctx::B200Context, Y, kind::Int, st, trim::Float64, trimmed::Bool)
    attach!(ctx, Y)
    out = Ref{Float64}(0.0)
    check(ccall((:vbmf_b200_mctx_lower_bound, LIB), Cint, (Ptr{Void}, Cint, Ptr{Void}, Float64, Cint, Ref{Float64}),
                ctx.handle, kind, st, trim, trimmed, out))
    return out[]
end
lowerBound(ctx::B200Context, Y, p) = lower_bound(ctx, Y, p, 0.0, false)
lowerBoundTrimmed(ctx::B200Context, Y, p, trim = 1e-1) = lower_bound(ctx, Y, p, Float64(trim), true)
# the reference's signatures (src/vbmf_sparse.jl:435,478; src/vbmf_dual.jl:556,606)
lowerBound(Y::Array{Float64,2}, p::Union{vbmf_sparse_parameters,vbmf_dual_parameters}) = lowerBound(default_context(), Y, p)
lowerBoundTrimmed(Y::Array{Float64,2}, p::Union{vbmf_sparse_parameters,vbmf_dual_parameters}, trim = 1e-1) = lowerBoundTrimmed(default_context(), Y, p, trim)

end # module
