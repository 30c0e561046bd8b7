// Launcher interface of the fused small kernels of the VB loop (everything that is not one of the two GEMMs).
#pragma once
#include "common.cuh"

namespace vb {

enum Kind { KIND_DENSE = 0, KIND_SPARSE = 1, KIND_DUAL = 2, KIND_TRIAL = 3 };
// ARD groups of vec(A') for dual / trial: 0: h < H0;  1: h >= H0 and global row < M0;  2: h >= H0 and global row >= M0
// (vbmf_dual is the case M0 = M, src/vbmf_dual.jl:322-351; vbmf_trial src/vbmf_trial.jl:357-400)

// Plain-old-data view of one solver's device state, passed by value to kernels.
struct Dev {
    int kind;
    int L, ldB;          // rows of Y; leading dimension of the [H][ldB] column-major L x H buffers
    int Mloc, Mglob, moff;   // columns of Y in this shard / in total / global index of the first local column
    int H, H0, H1;       // rank; dual/trial: first group width H0, second H1 = H - H0; dense/sparse: H1 masked columns
    int M0;              // trial: global row split of the second column group (dual: = Mglob)
    int nlabels;
    Scalars* sc;
    const double* Y; int ldY;
    double* rowY2;       // [L] global sum_m Y[l,m]^2
    double* A;           // [Mloc][H]   AHat rows (== ATVecHat slice, H fastest)
    double* P;           // [Mloc][H]   Y' * BHat (raw K1 output / staging)
    double* B;           // [H][ldB]    BHat
    double* Bold;        // [H][ldB]    previous BHat
    double* D;           // [H][ldB]    BHat - Bold
    double* Bs;          // [H][ldB]    diag(sigmaVecHat) * BHat (diag_var)
    double* packed;      // [H*ldB | H*H | H*H | 8]  all-reduce payload: Q, A'A, sum of Sigma blocks, dual sums
    double* SigmaA; double* SigmaB;           // [H][H]
    double* CA; double* CB; double* invCA; double* invCB;   // dense: [H][H]
    double* CAv; double* beta; double* sdiag; // sparse/dual: [Mloc*H] prior precision, its rate, diag of Sigma
    double* blocks;      // optional [Mloc][H][H] full_cov covariance blocks (nullptr unless requested)
    double* CBv; double* deltav;              // sparse/dual: [H]
    double* sigmaVec; double* etaVec; double* zetaVec;   // [L]
    double* BtB; double* BtBw; double* DtD;   // [H][H] Grams: B'B, B'diag(w)B, D'D
    double* Gm;          // [H][H] likelihood part of the per-column precision (full_cov)
    double* part;        // partial-sum workspace
    const int* labels;   // local 0-based rows of A to mask
    const unsigned char* rowmask;   // [Mloc] 1 where the row is labelled (nullptr without labels)
    double* lbacc;       // [32] lower-bound accumulators
};

__host__ __device__ inline size_t packed_q(const Dev& d) { return 0; }
__host__ __device__ inline size_t packed_ata(const Dev& d) { return (size_t)d.H * d.ldB; }
__host__ __device__ inline size_t packed_sa(const Dev& d) { return (size_t)d.H * d.ldB + (size_t)d.H * d.H; }
__host__ __device__ inline size_t packed_ex(const Dev& d) { return (size_t)d.H * d.ldB + 2 * (size_t)d.H * d.H; }
__host__ __device__ inline size_t packed_len(const Dev& d) { return packed_ex(d) + 8; }

constexpr int MAX_PARTS = 592;   // upper bound on per-kernel partial blocks (4 x 148)

// ---- peer exchange over NVLink (world <= 8, H <= 64, homoscedastic): the all-reduce -> SigmaB -> BHat epilogue chain of
// updateB! as reduce-scatter + row-sharded epilogue + all-gather done by our own kernels through peer-mapped memory.
// Every rank owns one peer-visible buffer [flags | packed | BHat | rank partials]; the pointers below are the SAME regions of
// every rank's buffer as seen from this device (own entry = local address).
constexpr int PX_MAX_WORLD = 8;
constexpr int PX_NBAR = 512;                       // barrier slots (one per participating CTA index)
constexpr size_t PX_FLAG_BYTES = (size_t)PX_NBAR * PX_MAX_WORLD * sizeof(unsigned long long);
struct PxDev {
    int rank, W;
    unsigned long long epoch;                      // barriers of this launch use epoch + 1, epoch + 2, ...
    unsigned long long* flags[PX_MAX_WORLD];       // [PX_NBAR][PX_MAX_WORLD]: slot (b, src) is written by rank src only
    double* packed[PX_MAX_WORLD];                  // all-reduce payload of every rank (same layout as Dev::packed)
    double* B[PX_MAX_WORLD];                       // BHat of every rank
    double* gpart[PX_MAX_WORLD];                   // [W][2*H*H + 1]: slot r holds rank r's partial BtB | DtD | tr(B.*Q)
    double* small[PX_MAX_WORLD];                   // [2*H*H + 8]: every rank's local A'A | Sigma sums | group sums (send slot)
    unsigned long long* wait_ns;                   // profiling (may be NULL): [3][2] = {sum of wait ns, waits} of CTA 0 per barrier site
    int site;                                      // 0 small exchange, 1 epilogue, 2 Gram reduction
};

// flags shared by steps
enum {
    F_DIAG_VAR = 1, F_FULL_COV = 2, F_EST_CB = 4, F_EST_PRIORS = 8, F_EST_COVS = 16, F_EST_VAR = 32,
    F_FORCE = 64   // ignore sc->active (step-level API)
};

// opt the kernels of kernels.cu / batched.cu into their dynamic shared memory on the CURRENT device (once per context)
int kernels_init_device();

int k_set_control(cudaStream_t st, const Dev& d, int niter, double eps, int norm_mode, int force_active);
int k_y_stats(cudaStream_t st, const Dev& d, double* out_tr /*device, 1*/);
int k_transpose(cudaStream_t st, const double* src, double* dst, int rows, int cols);  // src col-major rows x cols -> dst row-major
int k_gram(cudaStream_t st, const Dev& d, const double* X, bool amat, int n, const double* w, double* out);
int k_gram_w2(cudaStream_t st, const Dev& d, const double* X, int n, const double* w, double* out);   // weights squared (Q4)
int k_trbq(cudaStream_t st, const Dev& d);                       // sc->trBQ = sum(BHat .* Q)
int k_mean_sigma(cudaStream_t st, const Dev& d);                 // sc->meanSigmaVec = mean(sigmaVecHat)
int k_total(cudaStream_t st, const double* x, int n, double* out);   // out[0] = sum(x), single CTA, fixed order
int k_norms_init(cudaStream_t st, const Dev& d);                 // normBold = norm(BHat) from d.BtB
int k_dense_sigmaA(cudaStream_t st, const Dev& d);               // SigmaA = sigma2*inv(B'B + L*SigmaB + sigma2*invCA)
int k_dense_A_fused(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride);   // A = (sum_s P_s * SigmaA)/sigma2, mask, A'A
int k_dense_A_fused_range(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride, int m_begin, int m_end,
                          int part_base, int max_parts, int* nparts);      // one column chunk; Gram partials stay in d.part
int k_sum_gram_partials(cudaStream_t st, const Dev& d, int nparts);       // packed.AtA = sum of the chunk partials
int k_y_stats_chunk(cudaStream_t st, const Dev& d, int m0, int n, int first);   // rowY2 (+)= row norms of one column chunk
int k_copy_trYTY(cudaStream_t st, const Dev& d, const double* d_tr);      // sc->trYTY = *d_tr (device side, stream ordered)
int k_sparse_A_diag(cudaStream_t st, const Dev& d, int flags);   // diagonal path incl. Q2 map; partial column sums of s
int k_sparse_A_full(cudaStream_t st, const Dev& d, int flags);   // batched H x H SPD inverse per column
int k_sparse_A_full_ex(cudaStream_t st, const Dev& d, int flags, const double* slabs, int S, size_t slab_stride, int fuse_ca);
bool k_sparse_A_full_can_fuse(const Dev& d);                     // tensor-core path in use (H <= 32): slab sum / updateCA! can be fused
// whole-loop diagonal path in one pass: slab sum, A, diag, mask, beta/CA (+ group sums), A'A, diag SigmaA -> packed
int k_sparse_A_diag_fused(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride, int flags, int* defer_parts = nullptr);
int k_sparse_diag_reduce(cudaStream_t st, const Dev& d, int nparts);   // the deferred reduction of the fused diagonal pass
int k_mask(cudaStream_t st, const Dev& d);
int k_update_CA(cudaStream_t st, const Dev& d, int sums_only = 0);   // sparse / dual element-wise ARD update (+ dual sums)
int k_sum_slabs(cudaStream_t st, const double* slabs, int S, size_t n, double* out, const Scalars* sc);   // out = sum_s slabs[s]
int k_reduce_q(cudaStream_t st, const Dev& d, const double* Qpart, int S);   // fixed-order split-K reduction -> packed.Q
int k_sigmaB(cudaStream_t st, const Dev& d, int flags);          // SigmaB (dense / sparse), also SigmaA <- packed.SA (sparse)
int k_B_epilogue(cudaStream_t st, const Dev& d, int flags);      // BHat, Bold, D, partial tr(B.*Q)
// Row split of the exchange epilogue: 32-row tiles [lo, hi) of rank `rank`, and the CTA count, which is the SAME on every rank
// (CTA b meets CTA b of the peers at the barrier; a CTA without a tile contributes a zero partial).
inline void px_tile_range(int L, int W, int rank, int* lo, int* hi, int* grid) {
    const int ntiles = (L + 31) / 32;
    *lo = (int)((long long)ntiles * rank / W);
    *hi = (int)((long long)ntiles * (rank + 1) / W);
    const int per = (ntiles + W - 1) / W;
    *grid = per < 1 ? 1 : (per > 296 ? 296 : per);
}
// peer exchange (world > 1), one barrier (epoch + 1) each:
// global A'A / Sigma sums / group sums on every rank (needs only the A side of the iteration: runs beside K2) ...
int k_px_small(cudaStream_t st, const Dev& d, const PxDev& px);
// ... the BHat epilogue on this rank's rows: Q rows summed over the peers, BHat rows written to every peer ...
// ... and the rank partials of the Grams exchanged and summed in rank order.  H <= 64 only.
int k_B_epilogue_px(cudaStream_t st, const Dev& d, int flags, const PxDev& px, int* nparts);
int k_B_reduce_px(cudaStream_t st, const Dev& d, const PxDev& px, int nparts);
int k_sigma_rows(cudaStream_t st, const Dev& d);                 // diag_var: zetaVec, sigmaVecHat, mean
int k_scale_B(cudaStream_t st, const Dev& d);                    // Bs = diag(sigmaVecHat) * BHat
int k_post(cudaStream_t st, const Dev& d, int flags, bool with_delta);   // CA/CB/sigma/prior updates (+ delta, loop control)
int k_updateCB_only(cudaStream_t st, const Dev& d);
int k_dense_cov_only(cudaStream_t st, const Dev& d, int which);  // 0: CA/invCA  1: CB/invCB
int k_sigma_only(cudaStream_t st, const Dev& d, int flags);
int k_prior_only(cudaStream_t st, const Dev& d, int which);      // 0..2 alpha of group 0..2, 3..5 beta of group 0..2
int k_yhat(cudaStream_t st, const Dev& d, double* out, int ldo); // YHat = BHat * AHat'
int k_lower_bound(cudaStream_t st, const Dev& d, double trim, int trimmed, int phase);
int k_synth(cudaStream_t st, double* Y, int ldY, int L, int Mloc, int moff, int rank, double noise, uint64_t seed);
int k_randn(cudaStream_t st, double* x, size_t n, uint64_t seed, uint64_t stream);

// N3: preprocess / scaleY on the resident shard (src/util.jl:36-87)
int k_row_pass(cudaStream_t st, double* Y, int ldY, int L, int M, int mode, const double* mu, const double* den, double* part, double* out);
int k_finish_stats(cudaStream_t st, double* v, int L, double n, int mode);
int k_compact_rows(cudaStream_t st, const double* Y, int ldY, double* out, int ldo, const int* rows, int Lnew, int M, double lambda);
int k_scale_all(cudaStream_t st, double* Y, size_t n, double lambda);

// K11: batched vbls! (csrc/batched.cu).  A problem whose whole state fits one CTA's shared memory runs in the
// one-CTA-per-problem kernel; a larger one runs in the wide kernel, one thread-block cluster of CS CTAs per problem.
struct BatchDesc {
    int nprob, L, H, H0, kind, niter, full_cov, Mmax;
    const int* moff;        // [nprob+1] column offsets into the packed per-column arrays
    const double* Y;        // [L][Mtot] column-major, problems concatenated
    const double* B;        // [nprob][L*H] column-major L x H
    const double* SigmaB;   // [nprob][H*H]
    double* A;              // [Mtot][H]   in: unused (vbls overwrites), out: AHat rows
    double* CA;             // [Mtot*H]    in/out
    double* beta;           // [Mtot*H]    out
    double* sdiag;          // [Mtot*H]    out
    double* SigmaA;         // [nprob][H*H] out
    double* blocks;         // [Mtot][H][H] out or nullptr
    double* YHat;           // [L][Mtot] out or nullptr
    double* scal;           // [nprob][16]: 0 sigmaHat 1 eta 2 zeta 3 zeta0 4 trYTY 5 alpha (sparse) | M0 (trial) 6 beta0 (sparse)
                            //              7 8 = prior (alpha, beta) of ARD group 0, 9 10 = group 1, 14 15 = group 2 (trial)
                            //              out: 0 sigmaHat 2 zeta 11 12 6 = alpha of groups 0 1 2, 13 fail
    int diag_var;           // heteroscedastic noise (src/vbmf_sparse.jl:176-247 diag_var branches, :309-316)
    double* sigmaVec;       // [nprob][L]  in/out  (diag_var)
    const double* etaVec;   // [nprob][L]  in      (diag_var)
    double* zetaVec;        // [nprob][L]  out     (diag_var)
    const int* plist;       // problem of each launched CTA (one-CTA kernel) or cluster (wide kernel)
    double* V;              // wide kernel: [Mtot][H] V = B'Y (diag_var: B'diag(sv)Y)
    double* rowv;           // wide kernel, diag_var: [nprob][1 + 8][L] = ||Y[l,:]||^2 | per-rank partials of Y[l,:]*(A*b_l)
};
struct BatchDenseDesc {
    int nprob, L, H, niter, Mmax;
    const int* moff;
    const double* Y;        // [L][Mtot]
    const double* B;        // [nprob][L*H]
    const double* SigmaB;   // [nprob][H*H]
    double* A;              // [Mtot][H] out
    double* SigmaA;         // [nprob][H*H] out
    double* icA;            // [nprob][H] in: diag(invCA), out: diag(invCA)
    double* cA;             // [nprob][H] out: diag(CA)
    double* YHat;           // [L][Mtot] out or nullptr
    double* scal;           // [nprob][16]
    const int* plist;       // as BatchDesc::plist
    double* V;              // wide kernel: [Mtot][H] V = B'Y
};
constexpr int BATCH_MAX_CLUSTER = 8;   // portable thread-block cluster size
// CTAs of the wide kernel per problem: 0 = the problem fits the one-CTA kernel, else 1, 2, 4 or 8; -1 = H out of range
int batched_cluster_size(int kind, int L, int H, int M);
// Launches over a batch whose problems are grouped by cluster size: plist[0, n[0]) one-CTA problems (largest M: Mmax0),
// then n[1], n[2], n[3], n[4] problems for CS = 1, 2, 4, 8.
int k_batched_vbls(cudaStream_t st, const BatchDesc& bd, const int (&n)[5], int Mmax0);
int k_batched_vbls_dense(cudaStream_t st, const BatchDenseDesc& bd, const int (&n)[5], int Mmax0);

}  // namespace vb
