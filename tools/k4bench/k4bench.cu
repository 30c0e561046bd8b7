// Stand-alone timing + correctness probe for K4 (per-column H x H SPD inverses of the full-covariance A update,
// src/vbmf_sparse.jl:178-202): links the library's kernels.o, drives k_sparse_A_full on synthetic ARD-like precisions and
// compares with a host long-double Gauss-Jordan.  Development tool, not part of the product path.
//   k4bench [H=32] [M=100000] [reps=20]
//   k4bench hxh <H> [reps=50]
#include "../../vbmatrixfactorization.jl_b200/csrc/kernels.cuh"
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <random>
#include <algorithm>

namespace vb {
void set_error(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); fprintf(stderr, "\n"); }
void count_launch() {}
}
using namespace vb;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)

static void inv_ld(const std::vector<double>& S, int H, std::vector<double>& out) {
    std::vector<long double> A(S.begin(), S.end());
    for (int k = 0; k < H; ++k) {
        const long double d = A[k * H + k];
        std::vector<long double> col(H);
        for (int i = 0; i < H; ++i) col[i] = A[i * H + k];
        for (int i = 0; i < H; ++i)
            for (int j = 0; j < H; ++j) {
                long double v;
                if (i == k) v = (j == k) ? -1.0L / d : col[j] / d;
                else if (j == k) v = col[i] / d;
                else v = A[i * H + j] - col[i] * col[j] / d;
                A[i * H + j] = v;
            }
    }
    out.resize((size_t)H * H);
    for (int e = 0; e < H * H; ++e) out[e] = (double)(-A[e]);
}

// k4bench hxh <H> [reps]: the single H x H inverse of the dense A update (SigmaA = sigma2*inv(B'B + L*SigmaB + sigma2*invCA))
static int bench_hxh(int H, int reps) {
    CK(cudaSetDevice(0));
    if (kernels_init_device()) return 1;
    const int L = 1000;
    std::mt19937_64 rng(777);
    std::normal_distribution<double> nd(0.0, 1.0);
    std::uniform_real_distribution<double> ud(0.0, 1.0);
    const size_t HH = (size_t)H * H;
    std::vector<double> B((size_t)(H + 7) * H), BtB(HH, 0.0), SB(HH, 0.0), iCA(HH, 0.0), S(HH), Si;
    for (auto& x : B) x = nd(rng);
    for (int a = 0; a < H; ++a) for (int b = 0; b < H; ++b) { double t = 0; for (int l = 0; l < H + 7; ++l) t += B[l * H + a] * B[l * H + b]; BtB[a * H + b] = t; }
    for (int a = 0; a < H; ++a) { SB[a * H + a] = 1e-3 * ud(rng); iCA[a * H + a] = pow(10.0, -2.0 + 10.0 * ud(rng)); }
    const double s2 = 0.37;
    for (size_t e = 0; e < HH; ++e) S[e] = BtB[e] + (double)L * SB[e] + s2 * iCA[e];
    inv_ld(S, H, Si);
    Dev d; memset(&d, 0, sizeof(d));
    d.kind = KIND_DENSE; d.L = L; d.ldB = L; d.Mloc = 10; d.Mglob = 10; d.H = H;
    Scalars hs; memset(&hs, 0, sizeof(hs)); hs.active = 1; hs.sigma2 = s2;
    double *dBtB, *dSB, *diCA, *dSA; Scalars* dsc;
    CK(cudaMalloc(&dBtB, HH * 8)); CK(cudaMalloc(&dSB, HH * 8)); CK(cudaMalloc(&diCA, HH * 8)); CK(cudaMalloc(&dSA, HH * 8)); CK(cudaMalloc(&dsc, sizeof(Scalars)));
    CK(cudaMemcpy(dBtB, BtB.data(), HH * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dSB, SB.data(), HH * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(diCA, iCA.data(), HH * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dsc, &hs, sizeof(hs), cudaMemcpyHostToDevice));
    d.sc = dsc; d.BtB = dBtB; d.SigmaB = dSB; d.invCA = diCA; d.SigmaA = dSA;
    cudaStream_t st; CK(cudaStreamCreate(&st));
    for (int w = 0; w < 3; ++w) if (k_dense_sigmaA(st, d)) return 1;
    CK(cudaStreamSynchronize(st));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, st));
    for (int w = 0; w < reps; ++w) if (k_dense_sigmaA(st, d)) return 1;
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; CK(cudaEventElapsedTime(&ms, e0, e1));
    std::vector<double> hSA(HH);
    CK(cudaMemcpy(hSA.data(), dSA, HH * 8, cudaMemcpyDeviceToHost));
    double err = 0, mx = 0;
    for (size_t e = 0; e < HH; ++e) { err = std::max(err, fabs(hSA[e] - s2 * Si[e])); mx = std::max(mx, fabs(s2 * Si[e])); }
    printf("{\"kernel\": \"hxh (k_dense_sigmaA)\", \"H\": %d, \"us_per_launch\": %.2f, \"rel_err\": %.3g}\n", H, ms / reps * 1e3, err / mx);
    return 0;
}

int main(int argc, char** argv) {
    if (argc > 2 && strcmp(argv[1], "hxh") == 0) return bench_hxh(atoi(argv[2]), argc > 3 ? atoi(argv[3]) : 50);
    const int H = argc > 1 ? atoi(argv[1]) : 32, M = argc > 2 ? atoi(argv[2]) : 100000, reps = argc > 3 ? atoi(argv[3]) : 20;
    if (H < 1 || H > 128 || M < 1 || reps < 1) { fprintf(stderr, "usage: k4bench [H=32] [M=100000] [reps=20] | k4bench hxh <H> [reps=50]\n"); return 2; }
    CK(cudaSetDevice(0));
    if (kernels_init_device()) return 1;
    const int L = 64, ldB = 64;
    std::mt19937_64 rng(12345);
    std::normal_distribution<double> nd(0.0, 1.0);
    std::uniform_real_distribution<double> ud(0.0, 1.0);
    // G = sigmaHat*(B'B): B is L x H
    std::vector<double> B((size_t)L * H), BtB((size_t)H * H, 0.0), CA((size_t)M * H), P((size_t)M * H);
    for (auto& x : B) x = nd(rng);
    for (int a = 0; a < H; ++a) for (int b = 0; b < H; ++b) { double s = 0; for (int l = 0; l < L; ++l) s += B[l * H + a] * B[l * H + b]; BtB[a * H + b] = s; }
    for (auto& x : CA) x = pow(10.0, -2.0 + 12.0 * ud(rng));       // ARD precisions 1e-2 .. 1e10
    for (auto& x : P) x = nd(rng);
    const double sigmaHat = 0.7;
    Dev d; memset(&d, 0, sizeof(d));
    d.kind = KIND_SPARSE; d.L = L; d.ldB = ldB; d.Mloc = M; d.Mglob = M; d.H = H; d.H0 = H; d.M0 = M;
    Scalars hs; memset(&hs, 0, sizeof(hs)); hs.active = 1; hs.sigmaHat = sigmaHat;
    const size_t MH = (size_t)M * H, HH = (size_t)H * H;
    const size_t part_elems = std::max<size_t>((size_t)2400 * HH, 16384);
    double *dA, *dP, *dCA, *dsd, *dGm, *dBtB, *dSB, *dpacked, *dpart; Scalars* dsc;
    CK(cudaMalloc(&dA, MH * 8)); CK(cudaMalloc(&dP, MH * 8)); CK(cudaMalloc(&dCA, MH * 8)); CK(cudaMalloc(&dsd, MH * 8));
    CK(cudaMalloc(&dGm, HH * 8)); CK(cudaMalloc(&dBtB, HH * 8)); CK(cudaMalloc(&dSB, HH * 8));
    CK(cudaMalloc(&dpacked, ((size_t)H * ldB + 2 * HH + 8) * 8)); CK(cudaMalloc(&dpart, part_elems * 8)); CK(cudaMalloc(&dsc, sizeof(Scalars)));
    CK(cudaMemcpy(dP, P.data(), MH * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dCA, CA.data(), MH * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dBtB, BtB.data(), HH * 8, cudaMemcpyHostToDevice)); CK(cudaMemset(dSB, 0, HH * 8));
    CK(cudaMemcpy(dsc, &hs, sizeof(hs), cudaMemcpyHostToDevice));
    d.sc = dsc; d.A = dA; d.P = dP; d.CAv = dCA; d.sdiag = dsd; d.Gm = dGm; d.BtB = dBtB; d.SigmaB = dSB; d.packed = dpacked; d.part = dpart;
    cudaStream_t st; CK(cudaStreamCreate(&st));
    for (int w = 0; w < 3; ++w) if (k_sparse_A_full(st, d, F_FULL_COV)) return 1;
    CK(cudaStreamSynchronize(st));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, st));
    for (int w = 0; w < reps; ++w) if (k_sparse_A_full(st, d, F_FULL_COV)) return 1;
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; CK(cudaEventElapsedTime(&ms, e0, e1));
    std::vector<double> hA(MH), hsd(MH), hSA(HH);
    CK(cudaMemcpy(hA.data(), dA, MH * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(hsd.data(), dsd, MH * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hSA.data(), dpacked + (size_t)H * ldB + HH, HH * 8, cudaMemcpyDeviceToHost));
    // reference on every column (host, long double): a_m, diag, sum of blocks
    double errA = 0, errD = 0, maxA = 0;
    std::vector<long double> SA(HH, 0.0L);
    std::vector<double> S(HH), Si;
    const int stride = M > 20000 ? 7 : 1;                  // full check of sum(Sigma_m) only when cheap
    for (int m = 0; m < M; m += 1) {
        if (stride > 1 && (m % stride) && m > 512) continue;
        for (int a = 0; a < H; ++a) for (int b = 0; b < H; ++b) S[a * H + b] = sigmaHat * BtB[a * H + b] + (a == b ? CA[(size_t)m * H + a] : 0.0);
        inv_ld(S, H, Si);
        for (int a = 0; a < H; ++a) {
            long double s = 0; for (int b = 0; b < H; ++b) s += (long double)(sigmaHat * Si[a * H + b]) * P[(size_t)m * H + b];
            errA = std::max(errA, fabs(hA[(size_t)m * H + a] - (double)s)); maxA = std::max(maxA, fabs((double)s));
            errD = std::max(errD, fabs(hsd[(size_t)m * H + a] - Si[a * H + a]) / Si[a * H + a]);
        }
        for (size_t e = 0; e < HH; ++e) SA[e] += Si[e];
    }
    double errS = -1.0;
    if (stride == 1) { double mx = 0; errS = 0; for (size_t e = 0; e < HH; ++e) { mx = std::max(mx, fabs((double)SA[e])); errS = std::max(errS, fabs(hSA[e] - (double)SA[e])); } errS /= mx; }
    int fail = 0; CK(cudaMemcpy(&hs, dsc, sizeof(hs), cudaMemcpyDeviceToHost)); fail = hs.chol_fail;
    const double per = ms / reps;
    printf("{\"kernel\": \"k_sparse_A_full\", \"H\": %d, \"M\": %d, \"ms_per_launch\": %.4f, \"inverses_per_s\": %.4g, "
           "\"gflops_2H3\": %.1f, \"rel_err_A\": %.3g, \"rel_err_diag\": %.3g, \"rel_err_sumSigma\": %.3g, \"chol_fail\": %d}\n",
           H, M, per, M / (per * 1e-3), 2.0 * H * H * H * M / (per * 1e-3) * 1e-9,
           errA / maxA, errD, errS, fail);
    return 0;
}
