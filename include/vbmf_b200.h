/* vbmf_b200 -- C ABI of the B200-native VB matrix-factorisation update loop.
 *
 * Drop-in boundary for the hot path of vitskvara/VBMatrixFactorization.jl (the `while` loops of vbmf!, vbmf_sparse!,
 * vbmf_dual! and the update!/lowerBound step functions they call).  A Julia `ccall` shim (julia/VBMatrixFactorizationB200.jl,
 * INTEGRATION.md) or any other FFI binds exactly these symbols.  Citations are file:line in the reference repository.
 *
 * Conventions
 *   - plain pointers and sizes only; all matrices are host memory in Julia layout (column-major, Float64), labels are
 *     1-based Int64 exactly as Julia passes them; the library copies in and out, device memory is owned by ctx/solver.
 *   - every function returns 0 on success, <0 on error; vbmf_b200_last_error() gives the message (thread-local).
 *     There is no CPU fallback: no CUDA device => error.
 *   - calls on one ctx are synchronous and not re-entrant.
 *   - sharding: one ctx per GPU/rank owns the columns [col_offset, col_offset + M_local) of Y and the matching rows of
 *     AHat and per-element vectors; BHat, SigmaB, CB, noise and hyper-prior scalars are replicated.  world == 1 is the
 *     single-GPU case.  One packed all-reduce (NCCL, double, sum) of [Y*AHat | AHat'AHat | sum Sigma_m | prior sums]
 *     is issued per iteration.
 */
#ifndef VBMF_B200_H
#define VBMF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vbmf_b200_ctx vbmf_b200_ctx;       /* one GPU: stream, communicator, resident shard of Y */
typedef struct vbmf_b200_solver vbmf_b200_solver; /* device-resident parameter state of one problem */

enum { VBMF_B200_DENSE = 0, VBMF_B200_SPARSE = 1, VBMF_B200_DUAL = 2, VBMF_B200_TRIAL = 3 };
enum { VBMF_B200_NORM_SPECTRAL = 0,   /* Julia 0.5 norm(::Matrix) in delta(), src/util.jl:27-29 (default) */
       VBMF_B200_NORM_FROBENIUS = 1 };
/* option bits (keyword arguments of vbmf!/vbmf_sparse!/vbmf_dual! and of the step functions) */
enum {
    VBMF_B200_DIAG_VAR = 1,    /* diag_var   src/vbmf_sparse.jl:345 */
    VBMF_B200_FULL_COV = 2,    /* full_cov   src/vbmf_sparse.jl:345 */
    VBMF_B200_EST_CB = 4,      /* est_cb     src/vbmf_sparse.jl:345 */
    VBMF_B200_EST_PRIORS = 8,  /* est_priors src/vbmf_dual.jl:456 */
    VBMF_B200_EST_COVS = 16,   /* est_covs   src/vbmf.jl:175 */
    VBMF_B200_EST_VAR = 32     /* est_var    src/vbmf.jl:176 */
};
/* step functions of the reference, callable one by one (examples/mil_util.jl:183-197 does exactly that) */
enum {
    VBMF_B200_STEP_UPDATE_A = 0,       /* updateA!       src/vbmf.jl:95, src/vbmf_sparse.jl:176, src/vbmf_dual.jl:216 */
    VBMF_B200_STEP_UPDATE_B = 1,       /* updateB!       src/vbmf.jl:109, src/vbmf_sparse.jl:254, src/vbmf_dual.jl:292 */
    VBMF_B200_STEP_UPDATE_CA = 2,      /* updateCA!      src/vbmf.jl:129, src/vbmf_sparse.jl:284, src/vbmf_dual.jl:322 */
    VBMF_B200_STEP_UPDATE_CB = 3,      /* updateCB!      src/vbmf.jl:141, src/vbmf_sparse.jl:295, src/vbmf_dual.jl:358 */
    VBMF_B200_STEP_UPDATE_SIGMA = 4,   /* updateSigma2!  src/vbmf.jl:153 / updateSigma! src/vbmf_sparse.jl:307, src/vbmf_dual.jl:370 */
    VBMF_B200_STEP_UPDATE_ALPHA00 = 5, /* updateAlpha00! src/vbmf_dual.jl:393 */
    VBMF_B200_STEP_UPDATE_ALPHA01 = 6, /* updateAlpha01! src/vbmf_dual.jl:417 */
    VBMF_B200_STEP_UPDATE_BETA00 = 7,  /* updateBeta00!  src/vbmf_dual.jl:408 */
    VBMF_B200_STEP_UPDATE_BETA01 = 8,  /* updateBeta01!  src/vbmf_dual.jl:432 */
    /* vbmf_trial numbers its three ARD groups 1..3 (src/vbmf_trial.jl:442-507): updateAlpha01!/02!/03! = ALPHA00/01/02 here */
    VBMF_B200_STEP_UPDATE_ALPHA02 = 9, /* updateAlpha03! src/vbmf_trial.jl:490 */
    VBMF_B200_STEP_UPDATE_BETA02 = 10  /* updateBeta03!  src/vbmf_trial.jl:505 */
};

/* `vbmf_parameters`, src/vbmf.jl:22-40.  M = number of columns of Y held by this ctx. */
typedef struct {
    int64_t L, M, H, H1;
    int64_t n_labels;
    const int64_t* labels;   /* 1-based rows of AHat (shard-local) */
    double* AHat;            /* M x H */
    double* BHat;            /* L x H */
    double* SigmaA;          /* H x H */
    double* SigmaB;          /* H x H */
    double* CA;              /* H x H */
    double* CB;              /* H x H */
    double* invCA;           /* H x H */
    double* invCB;           /* H x H */
    double sigma2;
    double* YHat;            /* L x M or NULL (not produced when NULL; src/vbmf.jl:120) */
} vbmf_b200_dense_state;

/* `vbmf_sparse_parameters`, src/vbmf_sparse.jl:47-90.  SigmaATVec / invSigmaATVec ((MH)x(MH), :55,:57) are block
 * diagonal and exposed as M blocks of H x H (block m column-major, blocks consecutive) or NULL. */
typedef struct {
    int64_t L, M, H, MH, H1;
    int64_t n_labels;
    const int64_t* labels;
    double* AHat;            /* M x H */
    double* ATVecHat;        /* MH   (= vec(AHat'), H fastest) */
    double* SigmaATVec_blocks;     /* M*H*H or NULL */
    double* diagSigmaATVec;  /* MH */
    double* SigmaA;          /* H x H */
    double* BHat;            /* L x H */
    double* SigmaB;          /* H x H */
    double* CA;              /* MH */
    double alpha0, beta0, alpha;
    double* beta;            /* MH */
    double* CB;              /* H */
    double gamma0, delta0, gamma;
    double* delta;           /* H */
    double sigmaHat, eta0, zeta0, eta, zeta;
    double* sigmaVecHat;     /* L */
    double* etaVec;          /* L */
    double* zetaVec;         /* L */
    double* YHat;            /* L x M or NULL */
    double trYTY;
} vbmf_b200_sparse_state;

/* `vbmf_dual_parameters`, src/vbmf_dual.jl:59-112 (H1 = H - H0). */
typedef struct {
    int64_t L, M, MH, H, H0, H1;
    double* AHat;            /* M x H */
    double* ATVecHat;        /* MH */
    double* SigmaATVec_blocks;     /* M*H*H or NULL */
    double* diagSigmaATVec;  /* MH */
    double* SigmaA;          /* H x H */
    double* A0Hat;           /* M x H0 */
    double* A1Hat;           /* M x H1 */
    double* BHat;            /* L x H */
    double* SigmaB;          /* H x H */
    double* CA;              /* MH, per-row interleave [CA0 block m ; CA1 block m] */
    double* alpha;           /* 2 = [alpha0, alpha1] */
    double* beta;            /* MH, interleaved like CA */
    double* CA0;             /* M*H0 */
    double alpha00, beta00, alpha0;
    double* beta0;           /* M*H0 */
    double* CA1;             /* M*H1 */
    double alpha01, beta01, alpha1;
    double* beta1;           /* M*H1 */
    double* CB;              /* H */
    double gamma0, delta0, gamma;
    double* delta;           /* H */
    double sigmaHat, eta0, zeta0, eta, zeta;
    double* sigmaVecHat;     /* L */
    double* etaVec;          /* L */
    double* zetaVec;         /* L */
    double* YHat;            /* L x M or NULL */
    double trYTY;
} vbmf_b200_dual_state;

/* `vbmf_trial_parameters`, src/vbmf_trial.jl:68-129 (unexported in the reference, used by examples/mil_util.jl:194,253-290):
 * three ARD groups: A1 = AHat[:, 1:H0], A2 = AHat[1:M0, H0+1:H], A3 = AHat[M0+1:M, H0+1:H].  M0 / M1 are GLOBAL row counts of
 * AHat (columns of Y); with sharding M is the local row count and the shard's rows are split by their global index. */
typedef struct {
    int64_t L, M, M0, M1, MH, H, H0, H1;
    double* AHat;            /* M x H */
    double* ATVecHat;        /* MH */
    double* SigmaATVec_blocks;     /* M*H*H or NULL */
    double* diagSigmaATVec;  /* MH */
    double* SigmaA;          /* H x H */
    double* A1Hat;           /* M x H0 */
    double* A2Hat;           /* (local rows with global index <= M0) x H1 */
    double* A3Hat;           /* (local rows with global index  > M0) x H1 */
    double* BHat;            /* L x H */
    double* SigmaB;          /* H x H */
    double* CA;              /* MH, per-row interleave [CA1 block m ; CA2 or CA3 block m] */
    double* alpha;           /* 3 = [alpha1, alpha2, alpha3] */
    double* beta;            /* MH, interleaved like CA */
    double* CA1;             /* M*H0 */
    double alpha01, beta01, alpha1;
    double* beta1;           /* M*H0 */
    double* CA2;             /* M0*H1 (local part) */
    double alpha02, beta02, alpha2;
    double* beta2;
    double* CA3;             /* M1*H1 (local part) */
    double alpha03, beta03, alpha3;
    double* beta3;
    double* CB;              /* H */
    double gamma0, delta0, gamma;
    double* delta;           /* H */
    double sigmaHat, eta0, zeta0, eta, zeta;
    double* sigmaVecHat;     /* L */
    double* etaVec;          /* L */
    double* zetaVec;         /* L */
    double* YHat;            /* L x M or NULL */
    double trYTY;
} vbmf_b200_trial_state;

/* ---- library ---- */
int vbmf_b200_version(void);
const char* vbmf_b200_last_error(void);
int vbmf_b200_device_count(void);

/* ---- context ---- */
/* 128-byte NCCL unique id for a multi-rank job: rank 0 calls this and sends the bytes to the other ranks. */
int vbmf_b200_nccl_unique_id(void* id128);
/* cuda_stream: a cudaStream_t to enqueue on (e.g. the caller's current stream) or NULL to create one. */
int vbmf_b200_ctx_create(int device, int rank, int world, const void* nccl_id128, void* cuda_stream, vbmf_b200_ctx** out);
int vbmf_b200_ctx_destroy(vbmf_b200_ctx* ctx);
/* Y: L x M_local column-major host matrix with leading dimension ldY (the argument `Y` of every reference function).
 * Large matrices (>= 2 chunks of VBMF_B200_ATTACH_CHUNK_MB, default 2048 MB) are uploaded ASYNCHRONOUSLY in column chunks: the
 * call returns while the copy is in flight, the first dense iteration then works through the chunks as they arrive and every
 * other consumer waits for the upload on the device.  The host buffer must stay valid and unmodified until a call that uses Y
 * (a run, a step that contracts with Y, trYTY, download_Y) or vbmf_b200_ctx_sync has returned. */
int vbmf_b200_attach_Y(vbmf_b200_ctx* ctx, const double* Y, int64_t L, int64_t M_local, int64_t ldY, int64_t M_global,
                       int64_t col_offset);
/* Declare the problem geometry without data, for the step functions that take no Y in the reference (updateCA!(params),
 * updateCB!(params), updateAlpha0x!, updateYHat!): solvers can be created, steps that contract with Y return an error. */
int vbmf_b200_set_shape(vbmf_b200_ctx* ctx, int64_t L, int64_t M_local, int64_t M_global, int64_t col_offset);
/* Low-rank-plus-noise Y generated on the device (Philox4x32-10, keyed by the global column so any sharding agrees). */
int vbmf_b200_synth_Y(vbmf_b200_ctx* ctx, int64_t L, int64_t M_local, int64_t M_global, int64_t col_offset, int rank,
                      double noise, uint64_t seed);
/* preprocess(Y, lambda) (src/util.jl:73-87 incl. scaleY :36-53) applied to the attached Y on the device: row-standardise over
 * ALL columns (all shards), |var| <= 1e-15 -> 1, |Y - mean| <= 1e-8 -> 0, drop rows with sum(abs) < 1e-5, multiply by lambda.
 * The resident Y is replaced (L may shrink); L_out = new row count, used_rows (capacity L, 1-based, may be NULL) = kept rows.
 * Solvers created before this call are invalid. */
int vbmf_b200_preprocess_Y(vbmf_b200_ctx* ctx, double lambda, int64_t* L_out, int64_t* used_rows);
int vbmf_b200_download_Y(vbmf_b200_ctx* ctx, double* Y_out, int64_t ldY);
int vbmf_b200_trYTY(vbmf_b200_ctx* ctx, double* out);          /* traceXTY(Y, Y), src/vbmf_sparse.jl:150 */
int vbmf_b200_ctx_sync(vbmf_b200_ctx* ctx);
/* instrumentation for bench.py: kernel launches issued so far; CUDA-event time of the K1/K2 launches when profiling is on */
int64_t vbmf_b200_launch_count(void);
/* Host-side work decomposition of the two contractions for an L x M_local shard and rank H on a GPU with num_sms SMs (pure
 * host logic, needs no device): out[0] = K1 split count over L, out[1] = 16-row k-blocks per K1 split, out[2] = K2 split
 * count over M_local, out[3] = columns per K2 split (multiple of 16), out[4] = CTAs per SM, out[5] = tile width BN.
 * (none in the reference: src/vbmf.jl:98,112 are single BLAS calls) */
int vbmf_b200_plan_contractions(int64_t L, int64_t M_local, int64_t H, int num_sms, int64_t* out6);
/* enable: 0 off, 1 time the K1 / K2 launches and the exchange, 3 also mark the segments of every iteration (a few more event
 * records on the stream: use it for diagnosis, not for headline numbers) */
int vbmf_b200_ctx_profile(vbmf_b200_ctx* ctx, int enable);
/* Host-side row split of the peer-exchange epilogue (pure host logic, needs no device): out[0], out[1] = the 32-row tiles
 * [lo, hi) of BHat that `rank` of `world` (1..8) reduces, updates and broadcasts, out[2] = CTAs per rank (the same on every
 * rank).  (none in the reference: src/vbmf.jl:112 is one BLAS call on one host) */
int vbmf_b200_px_plan(int64_t L, int world, int rank, int64_t* out3);
int vbmf_b200_ctx_profile_read(vbmf_b200_ctx* ctx, double* k1_ms, int64_t* k1_launches, double* k2_ms, int64_t* k2_launches);
int vbmf_b200_ctx_profile_read_allreduce(vbmf_b200_ctx* ctx, double* allreduce_ms, int64_t* allreduce_launches);
/* Where an iteration's time goes on the main stream while profiling is on (CUDA events between the launches): ms[t] / n[t] =
 * total time / count of segment t = 1 K1, 2 A epilogue (+updateCA!), 3 K2, 4 split-K reduction of Y*AHat, 5 exchange between
 * the shards, 6 SigmaB, 7 BHat epilogue, 8 Gram reduction; 9..11 = mean time (ms) CTA 0 waited at the three peer-exchange
 * barriers (small sums, epilogue, Gram reduction), 12..20 = phases of CTA 0 in the last exchange-epilogue / Gram-reduction
 * launch.  Returns the number of segments (cap >= that; 32 is enough), -1 on error. */
int vbmf_b200_ctx_profile_read_segments(vbmf_b200_ctx* ctx, double* ms, int64_t* n, int cap);
/* 1 when this context's updateB! exchange (src/vbmf.jl:109-113 across column shards) runs through peer-mapped memory over
 * NVLink with the library's own kernels (world 2..8 on one node, H <= 64, decided when the first solver is created; switched
 * off with VBMF_B200_NO_PX=1), 0 when it uses the NCCL all-reduce.  (none in the reference: it is one process on one host) */
int vbmf_b200_ctx_peer_exchange(vbmf_b200_ctx* ctx);

/* ---- K1 / K2 on their own (parity tests of the two contractions) ---- */
/* P (M_local x H, column-major) = Y' * B ;  B is L x H column-major.  src/vbmf.jl:98 */
int vbmf_b200_gemm_YtB(vbmf_b200_ctx* ctx, const double* B, int64_t H, double* P);
/* Q (L x H, column-major) = Y * A over this shard's columns;  A is M_local x H column-major.  src/vbmf.jl:112 */
int vbmf_b200_gemm_YA(vbmf_b200_ctx* ctx, const double* A, int64_t H, double* Q);

/* ---- device-resident solver ---- */
/* h_split: H1 (masked trailing columns) for dense/sparse, H0 for dual.  labels: shard-local, 1-based, may be NULL. */
int vbmf_b200_solver_create(vbmf_b200_ctx* ctx, int kind, int64_t H, int64_t h_split, int64_t n_labels,
                            const int64_t* labels, int keep_blocks, vbmf_b200_solver** out);
/* vbmf_trial solver: H0 = width of the first column group, M0_global = number of rows of AHat (columns of Y) in group 2 */
int vbmf_b200_solver_create_trial(vbmf_b200_ctx* ctx, int64_t H, int64_t H0, int64_t M0_global, int keep_blocks,
                                  vbmf_b200_solver** out);
int vbmf_b200_solver_destroy(vbmf_b200_solver* s);
int vbmf_b200_dense_upload(vbmf_b200_solver* s, const vbmf_b200_dense_state* st);
int vbmf_b200_dense_download(vbmf_b200_solver* s, vbmf_b200_dense_state* st);
int vbmf_b200_sparse_upload(vbmf_b200_solver* s, const vbmf_b200_sparse_state* st);
int vbmf_b200_sparse_download(vbmf_b200_solver* s, vbmf_b200_sparse_state* st);
int vbmf_b200_dual_upload(vbmf_b200_solver* s, const vbmf_b200_dual_state* st);
int vbmf_b200_dual_download(vbmf_b200_solver* s, vbmf_b200_dual_state* st);
int vbmf_b200_trial_upload(vbmf_b200_solver* s, const vbmf_b200_trial_state* st);
int vbmf_b200_trial_download(vbmf_b200_solver* s, vbmf_b200_trial_state* st);
/* one reference step function on the resident state */
int vbmf_b200_solver_step(vbmf_b200_solver* s, int step, int flags);
/* the while-loop of vbmf! (src/vbmf.jl:193-214), vbmf_sparse! (src/vbmf_sparse.jl:368-393), vbmf_dual!
 * (src/vbmf_dual.jl:480-513) with the convergence test on the device.  iters = iterations done, d = last delta. */
int vbmf_b200_solver_run(vbmf_b200_solver* s, int64_t niter, double eps, int flags, int norm_mode, int64_t* iters, double* d);
/* Run the loops of n solvers of ONE single-GPU context in lockstep, with one K1 and one K2 per iteration serving all of them
 * (the sum of their H at most 64).  Each member behaves as vbmf_b200_solver_run would with its own flags[i]:
 *   - the same updates, in the same order;
 *   - its own convergence test: iters[i] and d[i] come back per member;
 *   - a member that has stopped keeps its state while the others go on;
 *   - failed[i] = 1 when its posterior precision was not positive definite: NaN in its state, its loop ended.
 * A member's result depends only on its own uploaded state, the resident Y and the sum of the members' H (which fixes the
 * split-K plans): reordering the members or changing another member's data leaves it bit for bit the same, and a group of
 * one equals vbmf_b200_solver_run.  Refused: n < 1, a solver twice, solvers of different contexts, a context with world > 1
 * or the peer exchange, a context without Y, a sum of H above 64.
 * Returns -2 when any member failed and 0 otherwise; other errors as usual, with every member's state unchanged. */
int vbmf_b200_solver_run_group(int n, vbmf_b200_solver* const* solvers, const int* flags, int64_t niter, double eps,
                               int norm_mode, int64_t* iters, double* d, int* failed);
/* The same loop with the reference's per-iteration logging hook (`update_log!(log, params)` after every iteration when
 * logdir != "", src/vbmf.jl:206-208, src/vbmf_sparse.jl:385-387, src/vbmf_dual.jl:505-507; log format src/data_manip.jl:6-66):
 * after each iteration the device is synchronised and cb(user, s, iterations_done, d) runs on the calling thread; it may call
 * the *_download function of the solver's kind to fetch the fields it logs (small fields only at scale: pass NULL for YHat
 * and the blocks).  A non-zero return stops the loop early.  cb == NULL behaves like vbmf_b200_solver_run one iteration at a time. */
typedef int (*vbmf_b200_iter_callback)(void* user, vbmf_b200_solver* s, int64_t iterations_done, double d);
int vbmf_b200_solver_run_logged(vbmf_b200_solver* s, int64_t niter, double eps, int flags, int norm_mode,
                                vbmf_b200_iter_callback cb, void* user, int64_t* iters, double* d);
/* lowerBound (trimmed = 0) / lowerBoundTrimmed (trimmed = 1), src/vbmf_sparse.jl:435-489, src/vbmf_dual.jl:556-617 */
int vbmf_b200_solver_lower_bound(vbmf_b200_solver* s, double trim, int trimmed, double* out);
/* updateYHat!: YHat (L x M_local, leading dimension ld) = BHat*AHat', src/vbmf.jl:120 */
int vbmf_b200_solver_yhat(vbmf_b200_solver* s, double* YHat, int64_t ld);

/* ---- batched small problems (the MIL classification pattern) ---- */
/* vbls! (examples/mil_util.jl:179-203) for nprob independent problems in one call on the context's stream:
 * niter x { updateA!, updateCA!, updateSigma! } with BHat fixed, then updateYHat! -- what classify(...; class_alg="dual")
 * runs for every test bag and class model (examples/mil_util.jl:504-511; class_alg = "vbls" :470-478 for dense parameters).
 * kind = VBMF_B200_DENSE, _SPARSE, _DUAL or _TRIAL (the four branches of vbls!, :182-197); states[p] points to the matching
 * state struct of problem p, Y[p] to its L x states[p]->M matrix.  All problems share L, H (and H0); M (and M0) may differ.
 * flags: VBMF_B200_FULL_COV, VBMF_B200_DIAG_VAR (both ignored for dense).  Needs no attached Y.  Limits: H <= 64 for sparse / dual /
 * trial (H > 32 with full_cov inverts one column at a time with the whole CTA) and H <= 32 for dense.  Dense and sparse
 * problems with H1 > 0 and labels get AHat[labels, H-H1+1:H] = 0 after every A update, as updateA! does (H1 in 0..H and
 * labels 1-based within 1..M of their own problem, as solver creation requires, else an error naming the problem; H1 may
 * differ per problem); dual and trial states have no labels.  A dense problem's first SigmaA uses its whole invCA;
 * updateCA! then leaves invCA = inv(diagonal CA), so after niter >= 1 it comes back diagonal with zeros off the diagonal.
 * Dense problems need a diagonal CA (what vbmf_init creates and updateCA! maintains).
 * A problem whose whole state fits one
 * CTA's shared memory runs in a one-CTA-per-problem kernel (one launch for all of them); a larger one runs in the wide
 * kernel, one thread-block cluster of 1, 2, 4 or 8 CTAs per problem (one launch per cluster size), see
 * vbmf_b200_batched_plan. */
int vbmf_b200_batched_vbls(vbmf_b200_ctx* ctx, int kind, int64_t nprob, const double* const* Y, void* const* states,
                           int64_t niter, int flags);
/* How vbmf_b200_batched_vbls runs each problem of a batch (host only, needs no GPU): cluster_out[p] = 0 when problem p (M[p]
 * columns) fits the one-CTA kernel, else the cluster size 1, 2, 4 or 8 of the wide kernel: the smallest whose per-CTA column
 * share stays within a fixed bound, at most 8.  full_cov / diag_var are 0 or 1 (ignored for dense).  Fails for H out of range
 * (H <= 64, dense H <= 32), an unknown kind or M[p] < 1. */
int vbmf_b200_batched_plan(int kind, int64_t L, int64_t H, int full_cov, int diag_var, int64_t nprob, const int64_t* M,
                           int32_t* cluster_out);

/* lowerBound (trimmed = 0) / lowerBoundTrimmed (trimmed = 1) of nprob independent problems in one call, on the
 * context's stream; out[p] = the ELBO of problem p.  src/vbmf_sparse.jl:435-489, src/vbmf_dual.jl:556-617,
 * src/vbmf_trial.jl:630-697.  kind = VBMF_B200_SPARSE, _DUAL or _TRIAL (the dense kind has no lowerBound); states[p] and
 * Y[p] as for vbmf_b200_batched_vbls, with the same limits: one L, H (and H0) for all problems, 1 <= H <= 64, M >= 1.
 * Reads ATVecHat when it is set, else AHat, like the single solver's upload; trYTY comes from the state; labels play no part.
 * Needs no attached Y and leaves the context's resident Y and its solvers alone.  A state whose arithmetic gives NaN (e.g.
 * a negative beta) gives NaN for its own problem only.  Every problem is split over CTAs by its own M and H alone, so its
 * bound is the same bit for bit whatever batch it is in. */
int vbmf_b200_batched_lower_bound(vbmf_b200_ctx* ctx, int kind, int64_t nprob, const double* const* Y,
                                  void* const* states, double trim, int trimmed, double* out);
/* norm(Y[p] - BHat*AHat') of nprob independent problems in one call, out[p] per problem.  norm_mode =
 * VBMF_B200_NORM_SPECTRAL (Julia 0.5 norm(::Matrix), largest singular value) or VBMF_B200_NORM_FROBENIUS (vecnorm): the
 * residual norms of classify(...; class_alg = "vbls") (examples/mil_util.jl:470-492) and, divided by L*M, of class_alg =
 * "dual" (:519-533), without YHat.  kind = any of the four kinds; states[p] and Y[p] as for vbmf_b200_batched_vbls.  Reads
 * only L, M, H, BHat and AHat of each state and writes nothing to it.  One L and H (H >= 1) for all problems, M >= 1 each,
 * at most 2^31 columns in all, and min(L, M) <= 2048 per problem in spectral mode.  Needs no attached Y and leaves the
 * context's resident Y and its solvers alone.  A NaN or Inf in a problem's residual gives NaN (spectral) or what the sum
 * of squares gives (Frobenius) for that problem only; a problem's norm is the same bit for bit whatever batch it is in. */
int vbmf_b200_batched_residual_norm(vbmf_b200_ctx* ctx, int kind, int64_t nprob, const double* const* Y,
                                    void* const* states, int norm_mode, double* out);

/* ---- one-call drop-ins: upload + loop + updateYHat! + download ---- */
/* vbmf!(Y, params, niter; eps, est_covs, est_var)   src/vbmf.jl:175 */
int vbmf_b200_dense_run(vbmf_b200_ctx* ctx, vbmf_b200_dense_state* st, int64_t niter, double eps, int est_covs, int est_var,
                        int norm_mode, int64_t* iters, double* d);
/* vbmf_sparse!(Y, params, niter; eps, diag_var, full_cov, est_cb)   src/vbmf_sparse.jl:344 */
int vbmf_b200_sparse_run(vbmf_b200_ctx* ctx, vbmf_b200_sparse_state* st, int64_t niter, double eps, int diag_var,
                         int full_cov, int est_cb, int norm_mode, int64_t* iters, double* d);
/* vbmf_dual!(Y, params, niter; eps, diag_var, full_cov, est_priors, est_cb)   src/vbmf_dual.jl:455 */
int vbmf_b200_dual_run(vbmf_b200_ctx* ctx, vbmf_b200_dual_state* st, int64_t niter, double eps, int diag_var, int full_cov,
                       int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d);

/* vbmf_trial!(Y, params, niter; eps, diag_var, full_cov, est_priors, est_cb)   src/vbmf_trial.jl:528 */
int vbmf_b200_trial_run(vbmf_b200_ctx* ctx, vbmf_b200_trial_state* st, int64_t niter, double eps, int diag_var, int full_cov,
                        int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d);

/* ---- several GPUs from ONE host process ---- */
/* The reference is a single Julia process making plain calls (src/vbmf.jl:175,238; src/vbmf_sparse.jl:344; src/vbmf_dual.jl:455),
 * so the drop-in must reach the column-sharded path without one process per GPU.  A multi-device context owns one ordinary
 * context per device (communicators from ncclCommInitAll) and drives them with one host thread per device inside the library.
 * Y and the state structs are the caller's FULL-SIZE host arrays (M = all columns, global 1-based labels); the library splits
 * the columns contiguously (device i gets [offset_i, offset_i + n_i), near-equal) and scatters / gathers AHat and the
 * per-element vectors itself.  Results equal the single-device ones up to the summation order of the all-reduce.
 * devices == NULL: devices 0 .. ndev-1; ndev <= 0: all visible devices. */
typedef struct vbmf_b200_mctx vbmf_b200_mctx;
int vbmf_b200_mctx_create(int ndev, const int* devices, vbmf_b200_mctx** out);
int vbmf_b200_mctx_destroy(vbmf_b200_mctx* mctx);
int vbmf_b200_mctx_ndev(vbmf_b200_mctx* mctx);
/* borrow the context of device i (valid until mctx_destroy), e.g. for vbmf_b200_ctx_profile */
int vbmf_b200_mctx_ctx(vbmf_b200_mctx* mctx, int i, vbmf_b200_ctx** out);
/* column range of device i after attach / synth */
int vbmf_b200_mctx_shard(vbmf_b200_mctx* mctx, int i, int64_t* col_offset, int64_t* n_cols);
/* Y: L x M column-major host matrix (all columns); every device uploads its own column range in parallel */
int vbmf_b200_mctx_attach_Y(vbmf_b200_mctx* mctx, const double* Y, int64_t L, int64_t M, int64_t ldY);
int vbmf_b200_mctx_synth_Y(vbmf_b200_mctx* mctx, int64_t L, int64_t M, int rank, double noise, uint64_t seed);
int vbmf_b200_mctx_trYTY(vbmf_b200_mctx* mctx, double* out);
/* vbmf!, vbmf_sparse!, vbmf_dual!, vbmf_trial! on the attached Y: same arguments as the one-call drop-ins above */
int vbmf_b200_mctx_dense_run(vbmf_b200_mctx* mctx, vbmf_b200_dense_state* st, int64_t niter, double eps, int est_covs, int est_var,
                             int norm_mode, int64_t* iters, double* d);
int vbmf_b200_mctx_sparse_run(vbmf_b200_mctx* mctx, vbmf_b200_sparse_state* st, int64_t niter, double eps, int diag_var,
                              int full_cov, int est_cb, int norm_mode, int64_t* iters, double* d);
int vbmf_b200_mctx_dual_run(vbmf_b200_mctx* mctx, vbmf_b200_dual_state* st, int64_t niter, double eps, int diag_var, int full_cov,
                            int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d);
int vbmf_b200_mctx_trial_run(vbmf_b200_mctx* mctx, vbmf_b200_trial_state* st, int64_t niter, double eps, int diag_var, int full_cov,
                             int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d);
/* lowerBound / lowerBoundTrimmed of a full-size sparse / dual / trial state (kind = VBMF_B200_SPARSE / _DUAL / _TRIAL) */
int vbmf_b200_mctx_lower_bound(vbmf_b200_mctx* mctx, int kind, void* state, double trim, int trimmed, double* out);

#ifdef __cplusplus
}
#endif
#endif /* VBMF_B200_H */
