// The one device definition of lowerBound / lowerBoundTrimmed (src/vbmf_sparse.jl:435-489, src/vbmf_dual.jl:556-617,
// src/vbmf_trial.jl:630-697) after the streamed sums are in: the single-solver lb_final_kernel (kernels.cu) and the batched
// batched_lb_final_kernel (batched.cu) both call these, so the two paths cannot drift apart.
#pragma once
#include "kernels.cuh"

namespace vb {

__device__ inline double gammaELn_d(double a, double logb) { return digamma_pos(a) - logb; }

// normalEntropy(kron(SigmaB, eye(L))) with Julia's left-to-right Float64 determinant product emulated (Q7):
// LU with partial pivoting of SigmaB, u_aa each repeated L times.  H <= 128.
//   CTA = false: one thread, no barriers.
//   CTA = true:  every thread of the block calls it; thread 0 picks the pivot (first index of the strict maximum) and keeps the
//                running L*log|u|, the rows of the trailing update are spread over the block.  sh: >= 2 doubles of shared memory.
// Every element goes through the same operations in both modes (f = W[i,k]/u, W[i,j] -= f*W[k,j]), so the results agree bit
// for bit.  W: H*H scratch (shared memory in CTA mode).
template <bool CTA>
__device__ double normal_entropy_kron(const double* SigmaB, int H, int L, double* W, double* sh) {
    const double LOG_EPS0 = -744.4400719213812;          // log(4.9406564584124654e-324)
    const double LOG_MIN = LOG_EPS0 - 0.6931471805599453, LOG_MAX = 709.782712893384;
    const int t = CTA ? (int)threadIdx.x : 0, nt = CTA ? (int)blockDim.x : 1;
    for (int e = t; e < H * H; e += nt) W[e] = SigmaB[e];
    double sign = 1.0, run = 0.0;
    int state = 0;   // 0 finite, 1 zero, 2 inf
    for (int k = 0; k < H && state == 0; ++k) {
        if (CTA) __syncthreads();                        // the previous trailing update (and the copy) are complete
        double u = 0.0;
        if (t == 0) {
            int piv = k; double best = fabs(W[k * H + k]);
            for (int i = k + 1; i < H; ++i) if (fabs(W[i * H + k]) > best) { best = fabs(W[i * H + k]); piv = i; }
            if (piv != k) {
                for (int j = 0; j < H; ++j) { const double tmp = W[k * H + j]; W[k * H + j] = W[piv * H + j]; W[piv * H + j] = tmp; }
                if (L & 1) sign = -sign;
            }
            u = W[k * H + k];
            if (u == 0.0) state = 1;
            else {
                if (u < 0.0 && (L & 1)) sign = -sign;
                // the running product does not depend on the trailing update: settle it first, so that the other
                // threads learn in the same barrier whether the loop ends
                run += (double)L * log(fabs(u));
                if (run < LOG_MIN) state = 1; else if (run > LOG_MAX) state = 2;
            }
            if (CTA) { sh[0] = u; sh[1] = (double)state; }
        }
        if (CTA) { __syncthreads(); u = sh[0]; state = (int)sh[1]; }
        if (u == 0.0 || state != 0) break;               // the factorisation ends here: no trailing update is needed
        for (int i = k + 1 + t; i < H; i += nt) {
            const double f = W[i * H + k] / u;
            for (int j = k + 1; j < H; ++j) W[i * H + j] -= f * W[k * H + j];
        }
    }
    double logd;
    if (state == 1) logd = LOG_EPS0;
    else if (state == 2) logd = sign > 0 ? INFINITY : LOG_EPS0;
    else { logd = sign > 0 ? run : LOG_EPS0; if (logd < LOG_EPS0) logd = LOG_EPS0; }
    const double m = (double)L * H;
    return m / 2 + m / 2 * 1.8378770664093453 + 0.5 * logd;   // meaningful in thread 0 (CTA mode: sign / run live there)
}

// What the lower bound needs besides the scalars: the sums over the MH elements (acc[0..10], lb_partial_kernel's layout),
// tr(GA.*GB), tr(diag(CB)*GB), sum(CB), sum(log(delta)), tr(BHat'*(Y*AHat)) and normalEntropy(kron(SigmaB, I_L)).
struct LbInputs {
    int kind, H, H0, H1;
    double L, M, M0;         // M0: trial row split (dual: unused)
    const double* acc;
    double tGAGB, trCBGB, sumCB, sumLogDelta, trBQ, entropyB;
};

// The term assembly, term by term in the reference's order (Q7, Q8, Q13).
__device__ inline double lb_assemble(const Scalars* sc, const LbInputs& in) {
    const double ln2pi = 1.8378770664093453;
    const int H = in.H;
    const double L = in.L, M = in.M;
    const double* acc = in.acc;
    const double elnS = gammaELn_d(sc->eta, log(sc->zeta));
    const double psiG = digamma_pos(sc->gamma);
    const double elnD = H * psiG - in.sumLogDelta;
    const double MHk = acc[10];                             // params.MH (kept count when trimmed)
    double Lb = 0.0;
    Lb += -L * M / 2 * ln2pi + L * M / 2 * elnS;
    Lb += -sc->sigmaHat / 2 * (sc->trYTY - 2 * in.trBQ + in.tGAGB);
    if (in.kind == KIND_SPARSE) {
        const double psiA = digamma_pos(sc->alpha);
        const double elnB = MHk * psiA - acc[6];
        Lb += -MHk / 2 * ln2pi + 0.5 * elnB;
        Lb += -(0.5 * acc[8]);
        Lb += -L * H / 2 * ln2pi;
        Lb += L / 2 * elnD;
        Lb += -0.5 * in.trCBGB;
        Lb += sc->eta0 * log(sc->zeta0) - lgamma(sc->eta0);
        Lb += (sc->eta0 - 1) * elnS - sc->zeta0 * sc->sigmaHat;
        Lb += MHk * (sc->alpha0p * log(sc->beta0p) - lgamma(sc->alpha0p));
        Lb += (sc->alpha0p - 1) * elnB;
        Lb += -sc->beta0p * acc[7];
        Lb += H * (sc->gamma0 * log(sc->delta0) - lgamma(sc->gamma0));
        Lb += (sc->gamma0 - 1) * elnD;
        Lb += -sc->gamma0 * in.sumCB;                       // Q13
        Lb += MHk / 2 + MHk / 2 * ln2pi + 0.5 * acc[9];
        Lb += in.entropyB;
        Lb += sc->eta + log(sc->zeta) + lgamma(sc->eta) + (1 - sc->eta) * digamma_pos(sc->eta);
        Lb += MHk * (sc->alpha + lgamma(sc->alpha) + (1 - sc->alpha) * psiA) + acc[6];
    } else {
        // dual (src/vbmf_dual.jl:559-597): groups 0, 1; trial (src/vbmf_trial.jl:633-681): groups 0, 1, 2.  Group sums use the
        // untrimmed beta_g / CA_g vectors even in lowerBoundTrimmed (only CA, ATVecHat, diagSigmaATVec, MH are trimmed).
        const int ng = in.kind == KIND_TRIAL ? 3 : 2;
        const double Ng[3] = {M * in.H0, in.M0 * in.H1, (M - in.M0) * in.H1};
        const double ag[3] = {sc->alpha_g0, sc->alpha_g1, sc->alpha_g2};
        const double a0g[3] = {sc->alpha00, sc->alpha01, sc->alpha02};
        const double b0g[3] = {sc->beta00, sc->beta01, sc->beta02};
        double psig[3], elng[3];
        for (int g = 0; g < ng; ++g) { psig[g] = digamma_pos(ag[g]); elng[g] = Ng[g] * psig[g] - acc[g]; }
        Lb += -MHk / 2 * ln2pi + 0.5 * elng[0];
        for (int g = 1; g < ng; ++g) Lb += 0.5 * elng[g];
        Lb += -(0.5 * acc[8]);
        Lb += -L * H / 2 * ln2pi;
        Lb += L / 2 * elnD;
        Lb += -0.5 * in.trCBGB;
        Lb += sc->eta0 * log(sc->zeta0) - lgamma(sc->eta0);
        Lb += (sc->eta0 - 1) * elnS - sc->zeta0 * sc->sigmaHat;
        for (int g = 0; g < ng; ++g) {
            Lb += Ng[g] * (a0g[g] * log(b0g[g]) - lgamma(a0g[g]));
            Lb += (a0g[g] - 1) * elng[g];
            Lb += -b0g[g] * acc[3 + g];
        }
        Lb += H * (sc->gamma0 * log(sc->delta0) - lgamma(sc->gamma0));
        Lb += (sc->gamma0 - 1) * elnD;
        Lb += -sc->gamma0 * in.sumCB;
        Lb += MHk / 2 + MHk / 2 * ln2pi + 0.5 * acc[9];
        Lb += in.entropyB;
        Lb += sc->eta + log(sc->zeta) + lgamma(sc->eta) + (1 - sc->eta) * digamma_pos(sc->eta);
        for (int g = 0; g < ng; ++g) Lb += (Ng[g] > 0 ? Ng[g] * (ag[g] + lgamma(ag[g]) + (1 - ag[g]) * psig[g]) : 0.0) + acc[g];
    }
    Lb += H * (sc->gamma + lgamma(sc->gamma) + (1 - sc->gamma) * psiG) + in.sumLogDelta;
    return Lb;
}

// The 11 sums of one element (lb_partial_kernel's layout): g = ARD group, av = AHat element, be = beta, ca = CA, s = diag Sigma.
__device__ __forceinline__ void lb_accumulate(double (&a)[11], int g, double av, double be, double ca, double s, double trim, int trimmed) {
    const double lbv = log(be);
    if (g == 0) { a[0] += lbv; a[3] += ca; } else if (g == 1) { a[1] += lbv; a[4] += ca; } else { a[2] += lbv; a[5] += ca; }
    if (!trimmed || fabs(av) > trim) {
        a[6] += lbv; a[7] += ca; a[8] += ca * (av * av + s); a[9] += log(s); a[10] += 1.0;
    }
}

}  // namespace vb
