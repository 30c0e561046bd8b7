// K11: `vbls!` for many small independent problems, one CTA per problem, one launch for the whole batch.
//
// Reference call pattern: examples/mil_util.jl:179-203 (vbls!: niter x { updateA!, updateCA!, updateSigma! } with BHat fixed,
// then updateYHat!) as used by classify(..., class_alg = "dual"/"vbls") (:453-535) on every test bag and every class model:
// thousands of L x M_p problems with L ~ 40, M_p = 5..40, H ~ 20.  With BHat fixed, B'B, B'Y and sum(Y.^2) are loop
// invariants, so the whole state of a problem lives in shared memory and registers for all niter iterations.
// Formulas: src/vbmf_sparse.jl:176-247 (updateA!, both covariance modes incl. Q2/Q3), :284-288 (updateCA!), :317-322
// (updateSigma!, homoscedastic); src/vbmf_dual.jl:322-351 for the two-group ARD update.
#include "kernels.cuh"
#include "linalg.cuh"
#include <algorithm>
#include <cooperative_groups.h>
#include <cstdlib>

namespace vb {

// HP = H rounded up to 8 / 16 / 24 / 32 for the warp-per-column register inverse; HP = 0: H > 32, the per-column inverses of
// the full-covariance path use the whole CTA on one shared-memory matrix (linalg.cuh::spd_inverse).
template <int HP>
__global__ void __launch_bounds__(128, (HP == 0 ? 1 : 3)) batched_vbls_kernel(BatchDesc bd) {
    extern __shared__ __align__(16) double sm[];
    __shared__ double red[32];
    __shared__ double s_sig, s_fail, s_msv;
    const int p = bd.plist[blockIdx.x];
    const int L = bd.L, H = bd.H, H0 = bd.H0;
    const int m0 = bd.moff[p], M = bd.moff[p + 1] - m0;
    const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, warp = t >> 5, nw = nt >> 5;
    const bool dvar = bd.diag_var != 0;
    // shared layout
    double* Bs = sm;                         // [L][H]
    double* V = Bs + L * H;                  // [M][H]   V[m][h] = (B'Y)[h][m]   (diag_var: (B'diag(sv)Y)[h][m])
    double* As = V + bd.Mmax * H;            // [M][H]
    double* CAs = As + bd.Mmax * H;          // [M][H]
    double* Ss = CAs + bd.Mmax * H;          // [M][H]   diag of Sigma
    double* G0 = Ss + bd.Mmax * H;           // [H][H]   B'B + L*SigmaB   (diag_var: B'diag(sv)B + L*mean(sv)*SigmaB)
    double* SA = G0 + H * H;                 // [H][H]
    double* AtA = SA + H * H;                // [H][H]
    double* dB = AtA + H * H;                // [H]      diag(B'B)        (diag_var: sum_l (B[l,h]*sv_l)^2, Q4)
    double* svs = dB + H;                    // [L]      sigmaVecHat
    double* ry2 = svs + L;                   // [L]      ||Y[l,:]||^2
    double* wrk = ry2 + L;                   // HP > 0: [nw][H*H + 98] per-warp sums of Sigma_m, column / p buffers
    wrk += (wrk - sm) & 1;                   //         (16-byte aligned: the register inverse reads them as double2)
                                             // HP == 0: [H][H+1] + 3H   the matrix being inverted + scratch
    double* scal = bd.scal + (size_t)p * 16;
    const double* Y = bd.Y + (size_t)m0 * L;
    const double* Bg = bd.B + (size_t)p * L * H;
    const double* SBg = bd.SigmaB + (size_t)p * H * H;

    for (int e = t; e < L * H; e += nt) { const int h = e / L, l = e - h * L; Bs[l * H + h] = Bg[e]; }
    for (int e = t; e < M * H; e += nt) CAs[e] = bd.CA[(size_t)m0 * H + e];
    for (int l = t; l < L; l += nt) {
        svs[l] = dvar ? bd.sigmaVec[(size_t)p * L + l] : 1.0;
        double s = 0.0;
        if (dvar) for (int m = 0; m < M; ++m) { const double y = Y[(size_t)m * L + l]; s = fma(y, y, s); }
        ry2[l] = s;
    }
    if (t == 0) { s_sig = scal[0]; s_fail = 0.0; }
    __syncthreads();
    // ARD groups (src/vbmf_dual.jl:322-351, src/vbmf_trial.jl:357-400): 0 = columns h < H0, 1 = h >= H0 and row m < M0,
    // 2 = h >= H0 and m >= M0 (trial only; dual has M0 = M, sparse H0 = H)
    const bool grouped = bd.kind == KIND_DUAL || bd.kind == KIND_TRIAL;
    const int M0p = bd.kind == KIND_TRIAL ? (int)scal[5] : M;
    const double eta = scal[1], zeta0 = scal[3], trYTY = scal[4];
    const double al0 = grouped ? scal[7] + 0.5 : scal[5], al1 = grouped ? scal[9] + 0.5 : scal[5], al2 = scal[14] + 0.5;
    const double be0 = grouped ? scal[8] : scal[6], be1 = grouped ? scal[10] : scal[6], be2 = scal[15];
    double zeta = scal[2];

    for (int it = 0; it < bd.niter; ++it) {
        // ---- loop invariants of the homoscedastic case are per-iteration quantities with diag_var: G0, diag(B'B), V
        if (it == 0 || dvar) {
            if (dvar) {
                double s = 0.0;
                for (int l = t; l < L; l += nt) s += svs[l];
                s = block_sum(s, red);
                if (t == 0) s_msv = s / (double)L;
                __syncthreads();
            }
            const double lw = dvar ? (double)L * s_msv : (double)L;
            for (int e = t; e < H * H; e += nt) {
                const int a = e / H, b = e - a * H;
                double s = 0.0, s2 = 0.0;
                for (int l = 0; l < L; ++l) {
                    const double w = svs[l], x = Bs[l * H + a];
                    s = fma(w * x, Bs[l * H + b], s);
                    if (a == b) s2 = fma(w * x, w * x, s2);
                }
                G0[e] = s + lw * SBg[e];
                if (a == b) dB[a] = dvar ? s2 : s;
            }
            for (int e = t; e < M * H; e += nt) {
                const int m = e / H, h = e - m * H;
                double s = 0.0;
                for (int l = 0; l < L; ++l) s = fma(svs[l] * Y[(size_t)m * L + l], Bs[l * H + h], s);
                V[e] = s;
            }
            __syncthreads();
        }
        const double sh = s_sig;
        const double gs = dvar ? 1.0 : sh;            // scale of G0 / of the right-hand side in updateA!
        // ---- updateA!
        if (bd.full_cov) {
            if constexpr (HP > 0) {
                const bool live = lane < H;
                double* wa = wrk + warp * (H * H + 98);    // this warp's running sum of Sigma_m (lane owns column `lane`)
                double* col = wa + H * H;
                col += (col - sm) & 1;
                double* pv = col + 64;
                if (live) for (int q = 0; q < H; ++q) wa[q * H + lane] = 0.0;
                bool all_ok = true;
                for (int m = warp; m < M; m += nw) {
                    const double ca = live ? CAs[m * H + lane] : 1.0;
                    double a[HP];
#pragma unroll
                    for (int q = 0; q < HP; ++q) a[q] = ((q < H && live) ? gs * G0[q * H + lane] : 0.0) + ((q == lane) ? ca : 0.0);
                    pv[lane] = live ? V[m * H + lane] : 0.0;
                    const bool ok = warp_spd_inverse_reg<HP>(a, (live ? gs * G0[lane * H + lane] : 0.0) + ca, lane, col);
                    all_ok = all_ok && ok;
                    double s = 0.0, dg = 0.0;
#pragma unroll
                    for (int q = 0; q < HP; ++q) {
                        s = fma(gs * a[q], pv[q], s);
                        if (q == lane) dg = a[q];
                    }
                    if (live) {
                        As[m * H + lane] = ok ? s : nan("");
                        Ss[m * H + lane] = ok ? dg : nan("");
                        if (bd.blocks != nullptr && it == bd.niter - 1) {
#pragma unroll
                            for (int q = 0; q < HP; ++q) if (q < H) bd.blocks[(size_t)(m0 + m) * H * H + q * H + lane] = a[q];
                        }
#pragma unroll
                        for (int q = 0; q < HP; ++q) if (q < H) wa[q * H + lane] += a[q];
                    }
                    __syncwarp();
                }
                if (!all_ok && lane == 0) s_fail = 1.0;
                __syncthreads();
                for (int e = t; e < H * H; e += nt) {
                    double s = 0.0;
                    for (int w = 0; w < nw; ++w) s += wrk[w * (H * H + 98) + e];
                    SA[e] = s;
                }
            } else {
                // H > 32: one column after the other, the whole CTA on one matrix
                BlockGroup g;
                const int ld = H + 1;
                double* Mx = wrk;
                double* vec = Mx + H * ld;
                for (int e = t; e < H * H; e += nt) SA[e] = 0.0;
                bool all_ok = true;
                for (int m = 0; m < M; ++m) {
                    __syncthreads();
                    for (int e = t; e < H * H; e += nt) { const int a = e / H, b = e - a * H; Mx[a * ld + b] = gs * G0[e] + (a == b ? CAs[m * H + a] : 0.0); }
                    __syncthreads();
                    const bool ok = spd_inverse(g, Mx, ld, H, vec);
                    all_ok = all_ok && ok;
                    for (int h = t; h < H; h += nt) {
                        double s = 0.0;
                        for (int k = 0; k < H; ++k) s = fma(gs * Mx[h * ld + k], V[m * H + k], s);
                        As[m * H + h] = ok ? s : nan("");
                        Ss[m * H + h] = ok ? Mx[h * ld + h] : nan("");
                    }
                    for (int e = t; e < H * H; e += nt) {
                        const double x = Mx[(e / H) * ld + (e % H)];
                        SA[e] += x;
                        if (bd.blocks != nullptr && it == bd.niter - 1) bd.blocks[(size_t)(m0 + m) * H * H + e] = x;
                    }
                }
                if (!all_ok && t == 0) s_fail = 1.0;
            }
        } else {
            // diagonal path incl. Q2: element j (0-based) reads d[j] for j < H, else d[(j - H) / (M - 1)]; Q3 / Q4 for d
            for (int e = t; e < M * H; e += nt) {
                const int src = (e < H) ? e : (e - H) / max(M - 1, 1);
                const double dsrc = dvar ? dB[src] + (double)L * s_msv * SBg[src * H + src] : sh * dB[src] + (double)L * SBg[src * H + src];
                const double s = 1.0 / (dsrc + CAs[e]);
                Ss[e] = s;
                As[e] = (gs * s) * V[e];
            }
            __syncthreads();
            for (int e = t; e < H * H; e += nt) {
                const int a = e / H, b = e - a * H;
                double s = 0.0;
                if (a == b) for (int m = 0; m < M; ++m) s += Ss[m * H + a];
                SA[e] = s;
            }
        }
        __syncthreads();
        // ---- updateCA!
        for (int e = t; e < M * H; e += nt) {
            const int m = e / H, h = e - m * H;
            const int g = (grouped && h >= H0) ? (m < M0p ? 1 : 2) : 0;
            const double a = As[e];
            const double beta = (g == 0 ? be0 : g == 1 ? be1 : be2) + 0.5 * (a * a + Ss[e]);
            CAs[e] = (g == 0 ? al0 : g == 1 ? al1 : al2) / beta;
            if (it == bd.niter - 1) bd.beta[(size_t)m0 * H + e] = beta;
        }
        // ---- updateSigma!
        for (int e = t; e < H * H; e += nt) {
            const int a = e / H, b = e - a * H;
            double s = 0.0;
            for (int m = 0; m < M; ++m) s = fma(As[m * H + a], As[m * H + b], s);
            AtA[e] = s;
        }
        if (dvar) {
            // per row l (src/vbmf_sparse.jl:309-316): zeta_l = zeta0 + ||Y[l,:]||^2/2 - Y[l,:]*(A*b_l) + traceXTY(A'A + SigmaA, b_l*b_l' + SigmaB)/2
            __syncthreads();
            double trc = 0.0;
            for (int e = t; e < H * H; e += nt) trc = fma(AtA[e] + SA[e], SBg[e], trc);
            trc = block_sum(trc, red);
            __syncthreads();
            if (t == 0) red[0] = trc;
            __syncthreads();
            trc = red[0];
            __syncthreads();
            for (int l = t; l < L; l += nt) {
                double qb = 0.0, quad = 0.0;
                for (int m = 0; m < M; ++m) {
                    double ab = 0.0;
                    for (int h = 0; h < H; ++h) ab = fma(As[m * H + h], Bs[l * H + h], ab);
                    qb = fma(Y[(size_t)m * L + l], ab, qb);
                }
                for (int a = 0; a < H; ++a) {
                    double row = 0.0;
                    for (int b = 0; b < H; ++b) row = fma(AtA[a * H + b] + SA[a * H + b], Bs[l * H + b], row);
                    quad = fma(Bs[l * H + a], row, quad);
                }
                const double z = zeta0 + 0.5 * ry2[l] - qb + 0.5 * (quad + trc);
                svs[l] = bd.etaVec[(size_t)p * L + l] / z;
                if (it == bd.niter - 1) bd.zetaVec[(size_t)p * L + l] = z;
            }
            __syncthreads();
        } else {
            // homoscedastic: G0 = B'B + L*SigmaB is exactly the second factor of the trace term (src/vbmf_sparse.jl:317-322)
            double tr = 0.0;
            for (int e = t; e < M * H; e += nt) tr = fma(V[e], As[e], tr);
            tr = block_sum(tr, red);            // leading __syncthreads also publishes AtA
            double tt = 0.0;
            for (int e = t; e < H * H; e += nt) tt = fma(AtA[e] + SA[e], G0[e], tt);
            __syncthreads();
            if (t == 0) red[0] = tr;
            __syncthreads();
            tr = red[0];
            tt = block_sum(tt, red);
            if (t == 0) {
                zeta = zeta0 + 0.5 * trYTY - tr + 0.5 * tt;
                s_sig = eta / zeta;
            }
            __syncthreads();
        }
    }
    // ---- outputs
    for (int e = t; e < M * H; e += nt) {
        bd.A[(size_t)m0 * H + e] = As[e];
        bd.CA[(size_t)m0 * H + e] = CAs[e];
        bd.sdiag[(size_t)m0 * H + e] = Ss[e];
    }
    for (int e = t; e < H * H; e += nt) bd.SigmaA[(size_t)p * H * H + e] = SA[e];
    if (dvar) for (int l = t; l < L; l += nt) bd.sigmaVec[(size_t)p * L + l] = svs[l];
    if (t == 0) { scal[0] = s_sig; scal[2] = zeta; scal[11] = al0; scal[12] = al1; scal[6] = al2; scal[13] = s_fail; }
    if (bd.YHat != nullptr) {   // updateYHat!  src/vbmf_sparse.jl:275
        for (int e = t; e < L * M; e += nt) {
            const int m = e / L, l = e - m * L;
            double s = 0.0;
            for (int h = 0; h < H; ++h) s = fma(Bs[l * H + h], As[m * H + h], s);
            bd.YHat[(size_t)(m0 + m) * L + l] = s;
        }
    }
}

size_t batched_smem_bytes(int L, int H, int Mmax, int nwarps) {
    const size_t work = H <= 32 ? (size_t)nwarps * (H * H + 98) + 2 : (size_t)H * (H + 1) + 3 * H;
    return (size_t)(L * H + 4 * Mmax * H + 3 * H * H + H + 2 * L + 2 + work) * sizeof(double) + 64;
}

// ---- wide problems: one thread-block cluster of CS CTAs per problem (CS = 1, 2, 4, 8)
// The problem's columns are split contiguously over the cluster ranks.  Per-column state (V, A, CA, diag Sigma) lives in
// global memory (the output arrays double as working storage), B is read from global memory, and the per-row vectors of
// diag_var (sigmaVecHat, ||Y[l,:]||^2, the partials of Y[l,:]*(A*b_l)) too; shared memory holds only H x H objects, so the
// footprint depends on H alone.  Cross-CTA sums (Sigma sums, A'A, trace, fail flag) go through distributed shared memory:
// every CTA writes its partial, and after a cluster barrier every CTA adds the partials of ranks 0, 1, ..., CS-1 in that
// order, so all ranks hold bit-identical totals and results do not change from run to run.
namespace cg = cooperative_groups;

__device__ __forceinline__ void cluster_sum(const cg::cluster_group& cl, int CS, double* part, double* out, int n) {
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < CS; ++r) s += cl.map_shared_rank(part, r)[e];
        out[e] = s;
    }
}

template <int HP>
__global__ void __launch_bounds__(128, (HP == 0 ? 1 : HP == 32 ? 2 : 3)) batched_vbls_wide_kernel(BatchDesc bd) {
    extern __shared__ __align__(16) double sm[];
    __shared__ double red[32];
    __shared__ double s_sig, s_fail, s_msv, s_tot[2];
    const cg::cluster_group cl = cg::this_cluster();
    const int CS = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int p = bd.plist[blockIdx.x / CS];
    const int L = bd.L, H = bd.H, H0 = bd.H0;
    const int m0 = bd.moff[p], M = bd.moff[p + 1] - m0;
    const int c0 = (int)((long long)M * rank / CS), nc = (int)((long long)M * (rank + 1) / CS) - c0;   // this CTA's columns
    const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, warp = t >> 5, nw = nt >> 5;
    const bool dvar = bd.diag_var != 0;
    double* G0 = sm;                         // [H][H]   as in batched_vbls_kernel
    double* SA = G0 + H * H;                 // [H][H]   cluster total
    double* AtA = SA + H * H;                // [H][H]   cluster total
    double* SAp = AtA + H * H;               // [H][H]   this CTA's partial (read by every rank)
    double* AtAp = SAp + H * H;              // [H][H]   this CTA's partial
    double* dB = AtAp + H * H;               // [H]
    double* sp = dB + H;                     // [2]      partial trace(V'A), partial fail flag
    double* wrk = sp + 2;
    wrk += (wrk - sm) & 1;
    double* scal = bd.scal + (size_t)p * 16;
    const size_t cb = (size_t)m0 + c0;       // first packed column of this CTA
    const double* Y = bd.Y + cb * L;
    const double* Bg = bd.B + (size_t)p * L * H;     // B[l, h] = Bg[h * L + l]
    const double* SBg = bd.SigmaB + (size_t)p * H * H;
    double* V = bd.V + cb * H;
    double* As = bd.A + cb * H;
    double* CAs = bd.CA + cb * H;
    double* Ss = bd.sdiag + cb * H;
    double* svs = dvar ? bd.sigmaVec + (size_t)p * L : nullptr;                        // rows l = rank (mod CS) are this CTA's
    double* ry2 = dvar ? bd.rowv + (size_t)p * (1 + BATCH_MAX_CLUSTER) * L : nullptr;
    double* qbp = dvar ? ry2 + L : nullptr;                                             // [CS][L]

    if (dvar) {
        const double* Yp = bd.Y + (size_t)m0 * L;
        for (int l = rank + t * CS; l < L; l += nt * CS) {
            double s = 0.0;
            for (int m = 0; m < M; ++m) { const double y = Yp[(size_t)m * L + l]; s = fma(y, y, s); }
            ry2[l] = s;
        }
    }
    if (t == 0) { s_sig = scal[0]; s_fail = 0.0; }
    __syncthreads();
    const bool grouped = bd.kind == KIND_DUAL || bd.kind == KIND_TRIAL;
    const int M0p = bd.kind == KIND_TRIAL ? (int)scal[5] : M;
    const double eta = scal[1], zeta0 = scal[3], trYTY = scal[4];
    const double al0 = grouped ? scal[7] + 0.5 : scal[5], al1 = grouped ? scal[9] + 0.5 : scal[5], al2 = scal[14] + 0.5;
    const double be0 = grouped ? scal[8] : scal[6], be1 = grouped ? scal[10] : scal[6], be2 = scal[15];
    double zeta = scal[2];

    for (int it = 0; it < bd.niter; ++it) {
        if (it == 0 || dvar) {
            if (dvar) {
                double s = 0.0;
                for (int l = t; l < L; l += nt) s += svs[l];
                s = block_sum(s, red);
                if (t == 0) s_msv = s / (double)L;
                __syncthreads();
            }
            const double lw = dvar ? (double)L * s_msv : (double)L;
            for (int e = t; e < H * H; e += nt) {
                const int a = e / H, b = e - a * H;
                double s = 0.0, s2 = 0.0;
                for (int l = 0; l < L; ++l) {
                    const double w = dvar ? svs[l] : 1.0, x = Bg[(size_t)a * L + l];
                    s = fma(w * x, Bg[(size_t)b * L + l], s);
                    if (a == b) s2 = fma(w * x, w * x, s2);
                }
                G0[e] = s + lw * SBg[e];
                if (a == b) dB[a] = dvar ? s2 : s;
            }
            for (int e = t; e < nc * H; e += nt) {
                const int m = e / H, h = e - m * H;
                double s = 0.0;
                for (int l = 0; l < L; ++l) s = fma((dvar ? svs[l] : 1.0) * Y[(size_t)m * L + l], Bg[(size_t)h * L + l], s);
                V[e] = s;
            }
            __syncthreads();
        }
        const double sh = s_sig;
        const double gs = dvar ? 1.0 : sh;
        // ---- updateA! on this CTA's columns; Sigma sums into SAp
        if (bd.full_cov) {
            if constexpr (HP > 0) {
                const bool live = lane < H;
                double* wa = wrk + warp * (H * H + 98);
                double* col = wa + H * H;
                col += (col - sm) & 1;
                double* pv = col + 64;
                if (live) for (int q = 0; q < H; ++q) wa[q * H + lane] = 0.0;
                bool all_ok = true;
                for (int m = warp; m < nc; m += nw) {
                    const double ca = live ? CAs[m * H + lane] : 1.0;
                    double a[HP];
#pragma unroll
                    for (int q = 0; q < HP; ++q) a[q] = ((q < H && live) ? gs * G0[q * H + lane] : 0.0) + ((q == lane) ? ca : 0.0);
                    pv[lane] = live ? V[m * H + lane] : 0.0;
                    const bool ok = warp_spd_inverse_reg<HP>(a, (live ? gs * G0[lane * H + lane] : 0.0) + ca, lane, col);
                    all_ok = all_ok && ok;
                    double s = 0.0, dg = 0.0;
#pragma unroll
                    for (int q = 0; q < HP; ++q) {
                        s = fma(gs * a[q], pv[q], s);
                        if (q == lane) dg = a[q];
                    }
                    if (live) {
                        As[m * H + lane] = ok ? s : nan("");
                        Ss[m * H + lane] = ok ? dg : nan("");
                        if (bd.blocks != nullptr && it == bd.niter - 1) {
#pragma unroll
                            for (int q = 0; q < HP; ++q) if (q < H) bd.blocks[(cb + m) * H * H + q * H + lane] = a[q];
                        }
#pragma unroll
                        for (int q = 0; q < HP; ++q) if (q < H) wa[q * H + lane] += a[q];
                    }
                    __syncwarp();
                }
                if (!all_ok && lane == 0) s_fail = 1.0;
                __syncthreads();
                for (int e = t; e < H * H; e += nt) {
                    double s = 0.0;
                    for (int w = 0; w < nw; ++w) s += wrk[w * (H * H + 98) + e];
                    SAp[e] = s;
                }
            } else {
                BlockGroup g;
                const int ld = H + 1;
                double* Mx = wrk;
                double* vec = Mx + H * ld;
                for (int e = t; e < H * H; e += nt) SAp[e] = 0.0;
                bool all_ok = true;
                for (int m = 0; m < nc; ++m) {
                    __syncthreads();
                    for (int e = t; e < H * H; e += nt) { const int a = e / H, b = e - a * H; Mx[a * ld + b] = gs * G0[e] + (a == b ? CAs[m * H + a] : 0.0); }
                    __syncthreads();
                    const bool ok = spd_inverse(g, Mx, ld, H, vec);
                    all_ok = all_ok && ok;
                    for (int h = t; h < H; h += nt) {
                        double s = 0.0;
                        for (int k = 0; k < H; ++k) s = fma(gs * Mx[h * ld + k], V[m * H + k], s);
                        As[m * H + h] = ok ? s : nan("");
                        Ss[m * H + h] = ok ? Mx[h * ld + h] : nan("");
                    }
                    for (int e = t; e < H * H; e += nt) {
                        const double x = Mx[(e / H) * ld + (e % H)];
                        SAp[e] += x;
                        if (bd.blocks != nullptr && it == bd.niter - 1) bd.blocks[(cb + m) * H * H + e] = x;
                    }
                }
                if (!all_ok && t == 0) s_fail = 1.0;
            }
        } else {
            // diagonal path; Q2's source index uses the element's index within the whole problem
            for (int e = t; e < nc * H; e += nt) {
                const int eg = c0 * H + e;
                const int src = (eg < H) ? eg : (eg - H) / max(M - 1, 1);
                const double dsrc = dvar ? dB[src] + (double)L * s_msv * SBg[src * H + src] : sh * dB[src] + (double)L * SBg[src * H + src];
                const double s = 1.0 / (dsrc + CAs[e]);
                Ss[e] = s;
                As[e] = (gs * s) * V[e];
            }
            __syncthreads();
            for (int e = t; e < H * H; e += nt) {
                const int a = e / H, b = e - a * H;
                double s = 0.0;
                if (a == b) for (int m = 0; m < nc; ++m) s += Ss[m * H + a];
                SAp[e] = s;
            }
        }
        __syncthreads();
        // ---- updateCA! (group split by the column index within the problem)
        for (int e = t; e < nc * H; e += nt) {
            const int m = e / H, h = e - m * H;
            const int g = (grouped && h >= H0) ? (c0 + m < M0p ? 1 : 2) : 0;
            const double a = As[e];
            const double beta = (g == 0 ? be0 : g == 1 ? be1 : be2) + 0.5 * (a * a + Ss[e]);
            CAs[e] = (g == 0 ? al0 : g == 1 ? al1 : al2) / beta;
            if (it == bd.niter - 1) bd.beta[cb * H + e] = beta;
        }
        // ---- partials of A'A and of the data term of updateSigma!
        for (int e = t; e < H * H; e += nt) {
            const int a = e / H, b = e - a * H;
            double s = 0.0;
            for (int m = 0; m < nc; ++m) s = fma(As[m * H + a], As[m * H + b], s);
            AtAp[e] = s;
        }
        double tr = 0.0;
        if (dvar) {
            for (int l = t; l < L; l += nt) {
                double qb = 0.0;
                for (int m = 0; m < nc; ++m) {
                    double ab = 0.0;
                    for (int h = 0; h < H; ++h) ab = fma(As[m * H + h], Bg[(size_t)h * L + l], ab);
                    qb = fma(Y[(size_t)m * L + l], ab, qb);
                }
                qbp[(size_t)rank * L + l] = qb;
            }
        } else {
            for (int e = t; e < nc * H; e += nt) tr = fma(V[e], As[e], tr);
        }
        tr = block_sum(tr, red);
        if (t == 0) { sp[0] = tr; sp[1] = s_fail; }
        cl.sync();
        cluster_sum(cl, CS, SAp, SA, H * H);
        cluster_sum(cl, CS, AtAp, AtA, H * H);
        cluster_sum(cl, CS, sp, s_tot, 2);
        cl.sync();                                     // every rank has read the partials before they are rewritten
        if (dvar) {
            double trc = 0.0;
            for (int e = t; e < H * H; e += nt) trc = fma(AtA[e] + SA[e], SBg[e], trc);
            trc = block_sum(trc, red);
            __syncthreads();
            if (t == 0) red[0] = trc;
            __syncthreads();
            trc = red[0];
            for (int l = rank + t * CS; l < L; l += nt * CS) {
                double qb = 0.0, quad = 0.0;
                for (int r = 0; r < CS; ++r) qb += qbp[(size_t)r * L + l];
                for (int a = 0; a < H; ++a) {
                    double row = 0.0;
                    for (int b = 0; b < H; ++b) row = fma(AtA[a * H + b] + SA[a * H + b], Bg[(size_t)b * L + l], row);
                    quad = fma(Bg[(size_t)a * L + l], row, quad);
                }
                const double z = zeta0 + 0.5 * ry2[l] - qb + 0.5 * (quad + trc);
                svs[l] = bd.etaVec[(size_t)p * L + l] / z;
                if (it == bd.niter - 1) bd.zetaVec[(size_t)p * L + l] = z;
            }
            cl.sync();                                 // the new sigmaVecHat rows are visible to every rank
        } else {
            double tt = 0.0;
            for (int e = t; e < H * H; e += nt) tt = fma(AtA[e] + SA[e], G0[e], tt);
            tt = block_sum(tt, red);
            if (t == 0) {
                zeta = zeta0 + 0.5 * trYTY - s_tot[0] + 0.5 * tt;
                s_sig = eta / zeta;
            }
            __syncthreads();
        }
    }
    // ---- outputs: A, CA, diag Sigma and sigmaVecHat are already in place
    if (rank == 0) {
        for (int e = t; e < H * H; e += nt) bd.SigmaA[(size_t)p * H * H + e] = SA[e];
        if (t == 0) { scal[0] = s_sig; scal[2] = zeta; scal[11] = al0; scal[12] = al1; scal[6] = al2; scal[13] = s_tot[1]; }
    }
    if (bd.YHat != nullptr) {
        for (int e = t; e < L * nc; e += nt) {
            const int m = e / L, l = e - m * L;
            double s = 0.0;
            for (int h = 0; h < H; ++h) s = fma(Bg[(size_t)h * L + l], As[m * H + h], s);
            bd.YHat[(cb + m) * L + l] = s;
        }
    }
}

size_t batched_wide_smem_bytes(int H, int nwarps) {
    const size_t work = H <= 32 ? (size_t)nwarps * (H * H + 98) + 2 : (size_t)H * (H + 1) + 3 * H;
    return (size_t)(5 * H * H + H + 2 + 1 + work) * sizeof(double) + 64;
}

static size_t batched_dense_smem_bytes(int L, int H, int Mmax) {
    return (size_t)(L * H + 2 * Mmax * H + 3 * H * H + 2 * H) * sizeof(double) + 64;
}

// Widest column share of one CTA of the wide kernel.  On the Musk2-shaped batch of tools/batched/large_bags.py (one B200)
// the kernels take 48 / 36 / 28 / 25 ms with bounds of 1e6 (cluster size 1 only) / 256 / 128 / 64 columns; the largest bag
// is the critical path.  VBMF_B200_BATCHED_COLS overrides the bound for such measurements.
static int batched_cols_per_cta() {
    static const int dflt = 64;
    const char* e = getenv("VBMF_B200_BATCHED_COLS");
    const int v = e ? atoi(e) : 0;
    return v > 0 ? v : dflt;
}

int batched_cluster_size(int kind, int L, int H, int M) {
    if (H < 1 || H > (kind == KIND_DENSE ? 32 : 64)) return -1;
    const int Lc = std::min(L, 1 << 20), Mc = std::min(M, 1 << 20);   // far beyond any budget; keeps the formulas in int
    const bool fits = kind == KIND_DENSE ? batched_dense_smem_bytes(Lc, H, Mc) <= 200 * 1024 : batched_smem_bytes(Lc, H, Mc, 4) <= 220 * 1024;
    if (fits) return 0;
    const int cols = batched_cols_per_cta();
    int cs = 1;
    while (cs < BATCH_MAX_CLUSTER && (M + cs - 1) / cs > cols) cs *= 2;
    return cs;
}

template <class D>
static int launch_wide(void (*kern)(D), const D& bd, int n, int CS, size_t smem, cudaStream_t st) {
    VB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n * CS));
    cfg.blockDim = dim3(128);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    VB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, bd));
    VB_LAUNCH_OK();
    return 0;
}

int k_batched_vbls(cudaStream_t st, const BatchDesc& bd, const int (&n)[5], int Mmax0) {
    if (bd.nprob <= 0) return 0;
    if (bd.H > 64) { set_error("batched vbls supports H <= 64 (got %d)", bd.H); return -1; }
    if (n[0] > 0) {
        BatchDesc b = bd;
        b.Mmax = Mmax0;
        const size_t smem = batched_smem_bytes(b.L, b.H, b.Mmax, 4);
#define BLAUNCH(HPV)                                                                                              \
    {                                                                                                             \
        VB_CUDA_OK(cudaFuncSetAttribute(batched_vbls_kernel<HPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        batched_vbls_kernel<HPV><<<n[0], 128, smem, st>>>(b);                                                     \
    }
        if (b.H <= 8) BLAUNCH(8) else if (b.H <= 16) BLAUNCH(16) else if (b.H <= 24) BLAUNCH(24) else if (b.H <= 32) BLAUNCH(32) else BLAUNCH(0)
#undef BLAUNCH
        VB_LAUNCH_OK();
    }
    const size_t wsmem = batched_wide_smem_bytes(bd.H, 4);
    for (int g = 1, off = n[0]; g < 5; off += n[g], ++g) {
        if (n[g] == 0) continue;
        BatchDesc b = bd;
        b.plist = bd.plist + off;
        const int CS = 1 << (g - 1);
        int rc;
        if (b.H <= 8) rc = launch_wide(batched_vbls_wide_kernel<8>, b, n[g], CS, wsmem, st);
        else if (b.H <= 16) rc = launch_wide(batched_vbls_wide_kernel<16>, b, n[g], CS, wsmem, st);
        else if (b.H <= 24) rc = launch_wide(batched_vbls_wide_kernel<24>, b, n[g], CS, wsmem, st);
        else if (b.H <= 32) rc = launch_wide(batched_vbls_wide_kernel<32>, b, n[g], CS, wsmem, st);
        else rc = launch_wide(batched_vbls_wide_kernel<0>, b, n[g], CS, wsmem, st);
        if (rc) return rc;
    }
    return 0;
}


// Dense `vbmf_parameters` flavour of vbls! (examples/mil_util.jl:182-185, the class_alg = "vbls" pattern :470-478):
//   updateA!      SigmaA = sigma2*inv(B'B + L*SigmaB + sigma2*invCA);  A = ((Y'B)*SigmaA)/sigma2        src/vbmf.jl:95-102
//   updateCA!     CA[h,h] = ||A[:,h]||^2/M + SigmaA[h,h];  invCA = inv(CA)                               src/vbmf.jl:129-134
//   updateSigma2! sigma2 = (sum(Y.^2) - 2*tr(Y'B A') + tr((A'A + M*SigmaA)(B'B + L*SigmaB)))/(L*M)       src/vbmf.jl:153-157
// One H x H inverse per iteration (warp 0, register-resident Gauss-Jordan); B'B, V = B'Y and sum(Y.^2) are loop invariants.
template <int HP>
__global__ void __launch_bounds__(128) batched_vbls_dense_kernel(BatchDenseDesc bd) {
    extern __shared__ __align__(16) double sm[];
    __shared__ double red[32];
    __shared__ __align__(16) double s_col[64];
    __shared__ double s_sig, s_fail;
    const int p = bd.plist[blockIdx.x];
    const int L = bd.L, H = bd.H;
    const int m0 = bd.moff[p], M = bd.moff[p + 1] - m0;
    const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, warp = t >> 5;
    double* Bs = sm;                         // [L][H]
    double* V = Bs + L * H;                  // [M][H]
    double* As = V + bd.Mmax * H;            // [M][H]
    double* G0 = As + bd.Mmax * H;           // [H][H]  B'B + L*SigmaB
    double* SA = G0 + H * H;                 // [H][H]
    double* AtA = SA + H * H;                // [H][H]
    double* ic = AtA + H * H;                // [H]     diag(invCA)
    double* cd = ic + H;                     // [H]     diag(CA)
    double* scal = bd.scal + (size_t)p * 16;
    const double* Y = bd.Y + (size_t)m0 * L;
    const double* Bg = bd.B + (size_t)p * L * H;
    const double* SBg = bd.SigmaB + (size_t)p * H * H;

    for (int e = t; e < L * H; e += nt) { const int h = e / L, l = e - h * L; Bs[l * H + h] = Bg[e]; }
    for (int e = t; e < H; e += nt) { ic[e] = bd.icA[(size_t)p * H + e]; cd[e] = 0.0; }
    if (t == 0) { s_sig = scal[0]; s_fail = 0.0; }
    double y2 = 0.0;
    for (int e = t; e < L * M; e += nt) { const double y = Y[e]; y2 = fma(y, y, y2); }
    y2 = block_sum(y2, red);                 // includes the barrier that publishes Bs
    __syncthreads();
    if (t == 0) red[0] = y2;
    __syncthreads();
    const double trYTY = red[0];
    __syncthreads();
    for (int e = t; e < H * H; e += nt) {
        const int a = e / H, b = e - a * H;
        double s = 0.0;
        for (int l = 0; l < L; ++l) s = fma(Bs[l * H + a], Bs[l * H + b], s);
        G0[e] = s + (double)L * SBg[e];
    }
    for (int e = t; e < M * H; e += nt) {
        const int m = e / H, h = e - m * H;
        double s = 0.0;
        for (int l = 0; l < L; ++l) s = fma(Y[(size_t)m * L + l], Bs[l * H + h], s);
        V[e] = s;
    }
    __syncthreads();
    for (int it = 0; it < bd.niter; ++it) {
        const double s2 = s_sig;
        // ---- updateA!: SigmaA
        if (warp == 0) {
            const bool live = lane < H;
            double a[HP];
#pragma unroll
            for (int q = 0; q < HP; ++q)
                a[q] = ((q < H && live) ? G0[q * H + lane] : 0.0) + ((q == lane) ? (live ? s2 * ic[lane] : 1.0) : 0.0);
            const double dg = live ? G0[lane * H + lane] + s2 * ic[lane] : 1.0;
            const bool ok = warp_spd_inverse_reg<HP>(a, dg, lane, s_col);
            if (live) {
#pragma unroll
                for (int q = 0; q < HP; ++q) if (q < H) SA[q * H + lane] = ok ? s2 * a[q] : nan("");
            }
            if (!ok && lane == 0) s_fail = 1.0;
        }
        __syncthreads();
        // ---- A = ((Y'B) * SigmaA) / sigma2
        for (int e = t; e < M * H; e += nt) {
            const int m = e / H, h = e - m * H;
            double s = 0.0;
            for (int k = 0; k < H; ++k) s = fma(V[m * H + k], SA[k * H + h], s);
            As[e] = s / s2;
        }
        __syncthreads();
        // ---- updateCA! and the Gram of A
        for (int e = t; e < H * H; e += nt) {
            const int a = e / H, b = e - a * H;
            double s = 0.0;
            for (int m = 0; m < M; ++m) s = fma(As[m * H + a], As[m * H + b], s);
            AtA[e] = s;
            if (a == b) { const double c = s / (double)M + SA[e]; cd[a] = c; ic[a] = 1.0 / c; }
        }
        // ---- updateSigma2!
        double tr = 0.0;
        for (int e = t; e < M * H; e += nt) tr = fma(V[e], As[e], tr);
        tr = block_sum(tr, red);            // leading barrier also publishes AtA
        __syncthreads();
        if (t == 0) red[0] = tr;
        __syncthreads();
        tr = red[0];
        __syncthreads();
        double tt = 0.0;
        for (int e = t; e < H * H; e += nt) tt = fma(AtA[e] + (double)M * SA[e], G0[e], tt);
        tt = block_sum(tt, red);
        if (t == 0) s_sig = (trYTY - 2.0 * tr + tt) / ((double)L * (double)M);
        __syncthreads();
    }
    for (int e = t; e < M * H; e += nt) bd.A[(size_t)m0 * H + e] = As[e];
    for (int e = t; e < H * H; e += nt) bd.SigmaA[(size_t)p * H * H + e] = SA[e];
    for (int e = t; e < H; e += nt) { bd.icA[(size_t)p * H + e] = ic[e]; bd.cA[(size_t)p * H + e] = cd[e]; }
    if (t == 0) { scal[0] = s_sig; scal[13] = s_fail; }
    if (bd.YHat != nullptr) {
        for (int e = t; e < L * M; e += nt) {
            const int m = e / L, l = e - m * L;
            double s = 0.0;
            for (int h = 0; h < H; ++h) s = fma(Bs[l * H + h], As[m * H + h], s);
            bd.YHat[(size_t)(m0 + m) * L + l] = s;
        }
    }
}

// Dense kind, wide problems: one cluster per problem as batched_vbls_wide_kernel.  A, V = B'Y in global memory; after the
// A'A reduction every CTA computes the H x H SigmaA inverse of the next iteration redundantly from identical inputs.
// SigmaA = sigma2*inv(G0 + sigma2*diag(ic)) by one warp; kept out of line so that the register-resident inverse does not
// share its register budget with the rest of the wide kernel
template <int HP>
__device__ __noinline__ bool dense_sigmaA_warp(const double* G0, const double* ic, double s2, double* SA, double* col, int H, int lane) {
    const bool live = lane < H;
    double a[HP];
#pragma unroll
    for (int q = 0; q < HP; ++q)
        a[q] = ((q < H && live) ? G0[q * H + lane] : 0.0) + ((q == lane) ? (live ? s2 * ic[lane] : 1.0) : 0.0);
    const double dg = live ? G0[lane * H + lane] + s2 * ic[lane] : 1.0;
    const bool ok = warp_spd_inverse_reg<HP>(a, dg, lane, col);
    if (live) {
#pragma unroll
        for (int q = 0; q < HP; ++q) if (q < H) SA[q * H + lane] = ok ? s2 * a[q] : nan("");
    }
    return ok;
}

template <int HP>
__global__ void __maxnreg__(255) batched_vbls_dense_wide_kernel(BatchDenseDesc bd) {
    extern __shared__ __align__(16) double sm[];
    __shared__ double red[32];
    __shared__ __align__(16) double s_col[64];
    __shared__ double s_sig, s_fail, s_tot[1];
    const cg::cluster_group cl = cg::this_cluster();
    const int CS = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int p = bd.plist[blockIdx.x / CS];
    const int L = bd.L, H = bd.H;
    const int m0 = bd.moff[p], M = bd.moff[p + 1] - m0;
    const int c0 = (int)((long long)M * rank / CS), nc = (int)((long long)M * (rank + 1) / CS) - c0;
    const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, warp = t >> 5;
    double* G0 = sm;                         // [H][H]  B'B + L*SigmaB
    double* SA = G0 + H * H;                 // [H][H]
    double* AtA = SA + H * H;                // [H][H]  cluster total
    double* AtAp = AtA + H * H;              // [H][H]  this CTA's partial
    double* ic = AtAp + H * H;               // [H]     diag(invCA)
    double* cd = ic + H;                     // [H]     diag(CA)
    double* sp = cd + H;                     // [1]     partial sum(Y.^2), then partial trace(V'A)
    double* scal = bd.scal + (size_t)p * 16;
    const size_t cb = (size_t)m0 + c0;
    const double* Y = bd.Y + cb * L;
    const double* Bg = bd.B + (size_t)p * L * H;
    const double* SBg = bd.SigmaB + (size_t)p * H * H;
    double* V = bd.V + cb * H;
    double* As = bd.A + cb * H;

    for (int e = t; e < H; e += nt) { ic[e] = bd.icA[(size_t)p * H + e]; cd[e] = 0.0; }
    if (t == 0) { s_sig = scal[0]; s_fail = 0.0; }
    double y2 = 0.0;
    for (int e = t; e < L * nc; e += nt) { const double y = Y[e]; y2 = fma(y, y, y2); }
    y2 = block_sum(y2, red);
    if (t == 0) sp[0] = y2;
    for (int e = t; e < H * H; e += nt) {
        const int a = e / H, b = e - a * H;
        double s = 0.0;
        for (int l = 0; l < L; ++l) s = fma(Bg[(size_t)a * L + l], Bg[(size_t)b * L + l], s);
        G0[e] = s + (double)L * SBg[e];
    }
    for (int e = t; e < nc * H; e += nt) {
        const int m = e / H, h = e - m * H;
        double s = 0.0;
        for (int l = 0; l < L; ++l) s = fma(Y[(size_t)m * L + l], Bg[(size_t)h * L + l], s);
        V[e] = s;
    }
    cl.sync();
    cluster_sum(cl, CS, sp, s_tot, 1);
    cl.sync();
    const double trYTY = s_tot[0];
    for (int it = 0; it < bd.niter; ++it) {
        const double s2 = s_sig;
        // ---- updateA!: SigmaA (identical on every rank)
        if (warp == 0 && !dense_sigmaA_warp<HP>(G0, ic, s2, SA, s_col, H, lane) && lane == 0) s_fail = 1.0;
        __syncthreads();
        // ---- A = ((Y'B) * SigmaA) / sigma2 on this CTA's columns
        for (int e = t; e < nc * H; e += nt) {
            const int m = e / H, h = e - m * H;
            double s = 0.0;
            for (int k = 0; k < H; ++k) s = fma(V[m * H + k], SA[k * H + h], s);
            As[e] = s / s2;
        }
        __syncthreads();
        for (int e = t; e < H * H; e += nt) {
            const int a = e / H, b = e - a * H;
            double s = 0.0;
            for (int m = 0; m < nc; ++m) s = fma(As[m * H + a], As[m * H + b], s);
            AtAp[e] = s;
        }
        double tr = 0.0;
        for (int e = t; e < nc * H; e += nt) tr = fma(V[e], As[e], tr);
        tr = block_sum(tr, red);
        if (t == 0) sp[0] = tr;
        cl.sync();
        cluster_sum(cl, CS, AtAp, AtA, H * H);
        cluster_sum(cl, CS, sp, s_tot, 1);
        cl.sync();
        // ---- updateCA! and updateSigma2! from the totals
        for (int a = t; a < H; a += nt) { const double c = AtA[a * H + a] / (double)M + SA[a * H + a]; cd[a] = c; ic[a] = 1.0 / c; }
        double tt = 0.0;
        for (int e = t; e < H * H; e += nt) tt = fma(AtA[e] + (double)M * SA[e], G0[e], tt);
        tt = block_sum(tt, red);
        if (t == 0) s_sig = (trYTY - 2.0 * s_tot[0] + tt) / ((double)L * (double)M);
        __syncthreads();
    }
    if (rank == 0) {
        for (int e = t; e < H * H; e += nt) bd.SigmaA[(size_t)p * H * H + e] = SA[e];
        for (int e = t; e < H; e += nt) { bd.icA[(size_t)p * H + e] = ic[e]; bd.cA[(size_t)p * H + e] = cd[e]; }
        if (t == 0) { scal[0] = s_sig; scal[13] = s_fail; }
    }
    if (bd.YHat != nullptr) {
        for (int e = t; e < L * nc; e += nt) {
            const int m = e / L, l = e - m * L;
            double s = 0.0;
            for (int h = 0; h < H; ++h) s = fma(Bg[(size_t)h * L + l], As[m * H + h], s);
            bd.YHat[(cb + m) * L + l] = s;
        }
    }
}

int k_batched_vbls_dense(cudaStream_t st, const BatchDenseDesc& bd, const int (&n)[5], int Mmax0) {
    if (bd.nprob <= 0) return 0;
    if (bd.H > 32) { set_error("batched vbls supports H <= 32 (got %d)", bd.H); return -1; }
    if (n[0] > 0) {
        BatchDenseDesc b = bd;
        b.Mmax = Mmax0;
        const size_t smem = batched_dense_smem_bytes(b.L, b.H, b.Mmax);
#define BDLAUNCH(HPV)                                                                                             \
    {                                                                                                             \
        VB_CUDA_OK(cudaFuncSetAttribute(batched_vbls_dense_kernel<HPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        batched_vbls_dense_kernel<HPV><<<n[0], 128, smem, st>>>(b);                                               \
    }
        if (b.H <= 8) BDLAUNCH(8) else if (b.H <= 16) BDLAUNCH(16) else if (b.H <= 24) BDLAUNCH(24) else BDLAUNCH(32)
#undef BDLAUNCH
        VB_LAUNCH_OK();
    }
    const size_t wsmem = (size_t)(4 * bd.H * bd.H + 2 * bd.H + 1) * sizeof(double) + 64;
    for (int g = 1, off = n[0]; g < 5; off += n[g], ++g) {
        if (n[g] == 0) continue;
        BatchDenseDesc b = bd;
        b.plist = bd.plist + off;
        const int CS = 1 << (g - 1);
        int rc;
        if (b.H <= 8) rc = launch_wide(batched_vbls_dense_wide_kernel<8>, b, n[g], CS, wsmem, st);
        else if (b.H <= 16) rc = launch_wide(batched_vbls_dense_wide_kernel<16>, b, n[g], CS, wsmem, st);
        else if (b.H <= 24) rc = launch_wide(batched_vbls_dense_wide_kernel<24>, b, n[g], CS, wsmem, st);
        else rc = launch_wide(batched_vbls_dense_wide_kernel<32>, b, n[g], CS, wsmem, st);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace vb
