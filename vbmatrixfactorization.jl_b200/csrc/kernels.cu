// Fused small kernels of the VB update loop: everything that is not one of the two contractions over Y.
// Every kernel is predicated on the device-side loop flag (Scalars::active) so iterations can be enqueued ahead of
// the device-side convergence test; every reduction uses a fixed order (per-CTA partials + ordered final sum).
// Reference formulas are cited per kernel (paths relative to /root/reference).
#include "kernels.cuh"
#include "elbo.cuh"
#include "linalg.cuh"
#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace vb {

#define ACTIVE_OR_RETURN(d) if (!(d).sc->active) return

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------- generic helpers
__global__ void sum_partials_kernel(const double* __restrict__ part, int nparts, size_t stride, size_t n,
                                    double* __restrict__ out, const Scalars* sc) {
    if (sc != nullptr && !sc->active) return;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        double s = 0.0;
#pragma unroll 8
        for (int p = 0; p < nparts; ++p) s += part[(size_t)p * stride + e];   // loads batched, sum order unchanged
        out[e] = s;
    }
}
// many partials, few outputs (Grams of per-CTA partials): 32 outputs x 8 partial-subsets per CTA, subsets combined in fixed
// order through shared memory -- 8x shorter dependent chains and n/32 CTAs instead of n/256
__global__ void __launch_bounds__(256) sum_partials_wide_kernel(const double* __restrict__ part, int nparts, size_t stride, size_t n,
                                                                double* __restrict__ out, const Scalars* sc) {
    if (sc != nullptr && !sc->active) return;
    __shared__ double sm[8][33];
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const size_t e = (size_t)blockIdx.x * 32 + x;
    double s = 0.0;
    if (e < n) {
#pragma unroll 4
        for (int p = y; p < nparts; p += 8) s += part[(size_t)p * stride + e];
    }
    sm[y][x] = s;
    __syncthreads();
    if (y == 0 && e < n) {
        double t = sm[0][x];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += sm[k][x];
        out[e] = t;
    }
}
static int sum_partials(cudaStream_t st, const double* part, int nparts, size_t stride, size_t n, double* out,
                        const Scalars* sc) {
    if (n == 0) return 0;
    if (nparts >= 16 && n <= (size_t)1 << 20) {
        sum_partials_wide_kernel<<<(unsigned)((n + 31) / 32), 256, 0, st>>>(part, nparts, stride, n, out, sc);
        VB_LAUNCH_OK();
        return 0;
    }
    int grid = std::max(1, std::min(cdiv((long)n, 256), 1184));
    sum_partials_kernel<<<grid, 256, 0, st>>>(part, nparts, stride, n, out, sc);
    VB_LAUNCH_OK();
    return 0;
}

__global__ void set_control_kernel(Scalars* sc, int niter, double eps, int norm_mode, int force_active) {
    sc->niter = niter;
    sc->eps = eps;
    sc->norm_mode = norm_mode;
    sc->iter = 0;
    sc->d = eps + 1.0;                                  // src/vbmf.jl:189  d = eps + 1.0
    sc->active = force_active ? 1 : ((1 <= niter) && (sc->d > eps)) ? 1 : 0;   // while (i <= niter) && (d > eps)
}
int k_set_control(cudaStream_t st, const Dev& d, int niter, double eps, int norm_mode, int force_active) {
    set_control_kernel<<<1, 1, 0, st>>>(d.sc, niter, eps, norm_mode, force_active);
    VB_LAUNCH_OK();
    return 0;
}

// col-major (rows x cols, ld = rows) -> row-major [rows][cols]
__global__ void transpose_kernel(const double* __restrict__ src, double* __restrict__ dst, int rows, int cols) {
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + threadIdx.x, c = c0 + i;
        if (r < rows && c < cols) tile[i][threadIdx.x] = src[(size_t)c * rows + r];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        if (r < rows && c < cols) dst[(size_t)r * cols + c] = tile[threadIdx.x][i];
    }
}
int k_transpose(cudaStream_t st, const double* src, double* dst, int rows, int cols) {
    if (rows <= 0 || cols <= 0) return 0;
    dim3 grid(cdiv(rows, 32), cdiv(cols, 32)), block(32, 8);
    transpose_kernel<<<grid, block, 0, st>>>(src, dst, rows, cols);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- K0: Y statistics
// trYTY = sum(Y.^2) (src/vbmf_sparse.jl:150; dense recomputes norm2(Y) every iteration, src/vbmf.jl:154) and the
// per-row ||Y[l,:]||^2 of the heteroscedastic update (src/vbmf_sparse.jl:310).
__global__ void y_stats_kernel(const double* __restrict__ Y, int ldY, int L, int M, int cols_per_blk, double* __restrict__ part) {
    const int m0 = blockIdx.y * cols_per_blk, m1 = min(M, m0 + cols_per_blk);
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    double s = 0.0;
    for (int m = m0; m < m1; ++m) { const double v = Y[(size_t)m * ldY + l]; s = fma(v, v, s); }
    part[(size_t)blockIdx.y * L + l] = s;
}
__global__ void total_kernel(const double* __restrict__ x, int n, double* out) {
    __shared__ double red[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += x[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s;
}
int k_total(cudaStream_t st, const double* x, int n, double* out) {
    total_kernel<<<1, 1024, 0, st>>>(x, n, out);
    VB_LAUNCH_OK();
    return 0;
}
// rowY2 (+)= per-row sum of squares of the columns [m0, m0 + n) (one upload chunk); chunks are accumulated in stream order
__global__ void accum_rows_kernel(const double* __restrict__ part, int nparts, int L, double* __restrict__ rowY2, int first) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    double s = first ? 0.0 : rowY2[l];
    for (int p = 0; p < nparts; ++p) s += part[(size_t)p * L + l];
    rowY2[l] = s;
}
int k_y_stats_chunk(cudaStream_t st, const Dev& d, int m0, int n, int first) {
    if (n <= 0 && !first) return 0;
    const int nby = std::max(1, std::min(MAX_PARTS / 2, cdiv(std::max(n, 1), 64)));
    const int cpb = cdiv(std::max(n, 1), nby);
    dim3 grid(cdiv(d.L, 128), nby);
    y_stats_kernel<<<grid, 128, 0, st>>>(d.Y + (size_t)m0 * d.ldY, d.ldY, d.L, n, cpb, d.part);
    VB_LAUNCH_OK();
    accum_rows_kernel<<<cdiv(d.L, 256), 256, 0, st>>>(d.part, nby, d.L, d.rowY2, first);
    VB_LAUNCH_OK();
    return 0;
}
__global__ void copy_tr_kernel(Scalars* sc, const double* d_tr) { sc->trYTY = d_tr[0]; }
int k_copy_trYTY(cudaStream_t st, const Dev& d, const double* d_tr) {
    copy_tr_kernel<<<1, 1, 0, st>>>(d.sc, d_tr);
    VB_LAUNCH_OK();
    return 0;
}
int k_y_stats(cudaStream_t st, const Dev& d, double* out_tr) {
    const int nby = std::max(1, std::min(MAX_PARTS / 2, cdiv(d.Mloc, 64)));
    const int cpb = cdiv(std::max(d.Mloc, 1), nby);
    dim3 grid(cdiv(d.L, 128), nby);
    y_stats_kernel<<<grid, 128, 0, st>>>(d.Y, d.ldY, d.L, d.Mloc, cpb, d.part);
    VB_LAUNCH_OK();
    // rowY2 (local); the caller all-reduces it across shards and totals again
    int g = std::max(1, std::min(cdiv(d.L, 256), 1184));
    sum_partials_kernel<<<g, 256, 0, st>>>(d.part, nby, (size_t)d.L, (size_t)d.L, d.rowY2, nullptr);
    VB_LAUNCH_OK();
    total_kernel<<<1, 1024, 0, st>>>(d.rowY2, d.L, out_tr);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- N3: preprocess / scaleY
// src/util.jl:36-53 (scaleY) and :73-87 (preprocess) on the resident shard: row mean and corrected variance over ALL columns
// (the caller all-reduces the per-row sums across shards), |var| <= 1e-15 -> 1, |Y - mu| <= 1e-8 -> 0, divide, then drop rows
// whose sum(abs) < 1e-5 and multiply by lambda.  mode 0: out[l] = sum_m Y   1: out[l] = sum_m (Y - mu_l)^2
// mode 2: Y <- scaled in place, out[l] = sum_m |Y_scaled|.  Fixed-order partials over column blocks.
__global__ void __launch_bounds__(128) row_pass_kernel(double* __restrict__ Y, int ldY, int L, int M, int cols_per_blk, int mode,
                                                       const double* __restrict__ mu, const double* __restrict__ den,
                                                       double* __restrict__ part) {
    const int m0 = blockIdx.y * cols_per_blk, m1 = min(M, m0 + cols_per_blk);
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    double s = 0.0;
    const double mul = mode ? mu[l] : 0.0, dl = (mode == 2) ? den[l] : 1.0;
    for (int m = m0; m < m1; ++m) {
        double* p = Y + (size_t)m * ldY + l;
        const double v = *p;
        if (mode == 0) s += v;
        else if (mode == 1) { const double c = v - mul; s = fma(c, c, s); }
        else {
            double c = v - mul;
            if (fabs(c) <= 1e-8) c = 0.0;
            c = c / dl;
            *p = c;
            s += fabs(c);
        }
    }
    part[(size_t)blockIdx.y * L + l] = s;
}
__global__ void finish_stats_kernel(double* mu_or_den, int L, double n, int mode) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    if (mode == 0) mu_or_den[l] = mu_or_den[l] / n;                 // mean(Y, 2)
    else {                                                          // var(Y, 2) -> guarded sqrt
        double d = mu_or_den[l] / (n - 1.0);
        if (fabs(d) <= 1e-15) d = 1.0;
        if (d == 0.0) d = 1.0;
        mu_or_den[l] = sqrt(d);
    }
}
// out[k, m] = lambda * Y[rows[k], m]   (row compaction into a fresh buffer)
__global__ void compact_rows_kernel(const double* __restrict__ Y, int ldY, double* __restrict__ out, int ldo, const int* __restrict__ rows,
                                    int Lnew, int M, double lambda) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y;
    if (k < Lnew && m < M) out[(size_t)m * ldo + k] = lambda * Y[(size_t)m * ldY + rows[k]];
}
__global__ void scale_all_kernel(double* Y, size_t n, double lambda) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) Y[i] *= lambda;
}
int k_row_pass(cudaStream_t st, double* Y, int ldY, int L, int M, int mode, const double* mu, const double* den, double* part, double* out) {
    const int nby = std::max(1, std::min(MAX_PARTS / 2, cdiv(std::max(M, 1), 64)));
    const int cpb = cdiv(std::max(M, 1), nby);
    dim3 grid(cdiv(L, 128), nby);
    row_pass_kernel<<<grid, 128, 0, st>>>(Y, ldY, L, M, cpb, mode, mu, den, part);
    VB_LAUNCH_OK();
    return sum_partials(st, part, nby, (size_t)L, (size_t)L, out, nullptr);
}
int k_finish_stats(cudaStream_t st, double* v, int L, double n, int mode) {
    finish_stats_kernel<<<cdiv(L, 256), 256, 0, st>>>(v, L, n, mode);
    VB_LAUNCH_OK();
    return 0;
}
int k_compact_rows(cudaStream_t st, const double* Y, int ldY, double* out, int ldo, const int* rows, int Lnew, int M, double lambda) {
    if (Lnew <= 0 || M <= 0) return 0;
    dim3 grid(cdiv(Lnew, 128), M);
    compact_rows_kernel<<<grid, 128, 0, st>>>(Y, ldY, out, ldo, rows, Lnew, M, lambda);
    VB_LAUNCH_OK();
    return 0;
}
int k_scale_all(cudaStream_t st, double* Y, size_t n, double lambda) {
    if (n == 0) return 0;
    scale_all_kernel<<<2368, 256, 0, st>>>(Y, n, lambda);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- Gram matrices
// G[a][b] = sum_i w_i^wpow X(i,a) X(i,b).  AMAT: X is [n][H] row-major (AHat rows); else X is [H][ld] (BHat-like).
// Used for BHat'BHat, AHat'AHat (src/vbmf.jl:96,110), B'diag(sv)B (src/vbmf_sparse.jl:182), norm2(B[:,h].*sv) (:211),
// D'D and Bold'Bold of the convergence test (src/util.jl:28).
template <int R, bool AMAT>
__global__ void __launch_bounds__(256) gram_partial_kernel(const double* __restrict__ X, int n, int H, int ld,
                                                           const double* __restrict__ w, int wpow, int rows_per_blk,
                                                           double* __restrict__ part, const Scalars* sc) {
    if (!sc->active) return;
    extern __shared__ double sm[];
    const int TS = H + 1;
    double* tile = sm;             // [32][TS]
    double* wt = sm + 32 * TS;     // [32]
    const int ta = threadIdx.x & 15, tb = threadIdx.x >> 4;
    double acc[R][R];
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) acc[i][j] = 0.0;
    const int r0 = blockIdx.x * rows_per_blk, r1 = min(n, r0 + rows_per_blk);
    for (int rt = r0; rt < r1; rt += 32) {
        const int nr = min(32, r1 - rt);
        __syncthreads();
        if (AMAT) {
            for (int e = threadIdx.x; e < 32 * H; e += 256) {
                const int i = e / H, a = e - i * H;
                tile[i * TS + a] = (i < nr) ? X[(size_t)(rt + i) * H + a] : 0.0;
            }
        } else {
            for (int e = threadIdx.x; e < 32 * H; e += 256) {
                const int a = e >> 5, i = e & 31;
                tile[i * TS + a] = (i < nr) ? X[(size_t)a * ld + rt + i] : 0.0;
            }
        }
        if (threadIdx.x < 32) {
            double wv = 1.0;
            if (w != nullptr && threadIdx.x < nr) { wv = w[rt + threadIdx.x]; if (wpow == 2) wv *= wv; }
            wt[threadIdx.x] = wv;
        }
        __syncthreads();
        for (int i = 0; i < 32; ++i) {
            double xa[R], xb[R];
            const double wv = wt[i];
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const int a = ta + 16 * q, b = tb + 16 * q;
                xa[q] = (a < H) ? tile[i * TS + a] * wv : 0.0;
                xb[q] = (b < H) ? tile[i * TS + b] : 0.0;
            }
#pragma unroll
            for (int p = 0; p < R; ++p)
#pragma unroll
                for (int q = 0; q < R; ++q) acc[p][q] = fma(xa[p], xb[q], acc[p][q]);
        }
    }
    double* out = part + (size_t)blockIdx.x * H * H;
#pragma unroll
    for (int p = 0; p < R; ++p)
#pragma unroll
        for (int q = 0; q < R; ++q) {
            const int a = ta + 16 * p, b = tb + 16 * q;
            if (a < H && b < H) out[a * H + b] = acc[p][q];
        }
}

// DMMA Gram: G = X'X over 32-row tiles staged in shared memory with the pitch-4 layout (see the A epilogue); accumulators
// in registers across the CTA's tiles, one partial per CTA.
__device__ __forceinline__ void dmma_acc2(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
__host__ __device__ inline int pitch4g(int hp8) { return ((hp8 + 11) / 16) * 16 + 4; }
template <int GT, bool AMAT>   // GT = upper-triangular 8x8 tiles per warp: ceil(nt8*(nt8+1)/2 / 8)
__global__ void __launch_bounds__(256) gram_dmma_kernel(const double* __restrict__ X, int n, int H, int ldx, double* __restrict__ part,
                                                        const Scalars* sc) {
    if (!sc->active) return;
    extern __shared__ double sm[];
    const int HP8 = (H + 7) & ~7, ld = pitch4g(HP8), nt8 = HP8 / 8;
    double* T = sm;     // [32][ld]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
    double g[GT][2];
    int gt[GT];           // this warp's tiles at | bt << 8 (at <= bt; the lower triangle is the bit-exact mirror), -1 = none
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        g[q][0] = 0.0; g[q][1] = 0.0;
        int idx = warp + 8 * q, at = 0;
        while (at < nt8 && idx >= nt8 - at) { idx -= nt8 - at; ++at; }
        gt[q] = at < nt8 ? (at | ((at + idx) << 8)) : -1;
    }
    const int ntiles = (n + 31) / 32;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int r0 = tile * 32, nr = min(32, n - r0);
        __syncthreads();
        if (AMAT) {
#pragma unroll 4
            for (int e = threadIdx.x; e < 32 * HP8; e += 256) {
                const int i = e / HP8, c = e - i * HP8;
                T[i * ld + c] = (i < nr && c < H) ? X[(size_t)(r0 + i) * H + c] : 0.0;
            }
        } else {
#pragma unroll 4
            for (int e = threadIdx.x; e < 32 * HP8; e += 256) {
                const int c = e >> 5, i = e & 31;
                T[i * ld + c] = (i < nr && c < H) ? X[(size_t)c * ldx + r0 + i] : 0.0;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < GT; ++q) {
            if (gt[q] >= 0) {
                const double* pa = T + j * ld + 8 * (gt[q] & 255) + r;
                const double* pb = T + j * ld + 8 * (gt[q] >> 8) + r;
#pragma unroll
                for (int i0 = 0; i0 < 32; i0 += 4) dmma_acc2(g[q], pa[i0 * ld], pb[i0 * ld]);
            }
        }
    }
    double* out = part + (size_t)blockIdx.x * H * H;
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        if (gt[q] >= 0) {
            const int a = 8 * (gt[q] & 255) + r, b = 8 * (gt[q] >> 8) + 2 * j;
            if (a < H && b < H) { out[a * H + b] = g[q][0]; out[b * H + a] = g[q][0]; }
            if (a < H && b + 1 < H) { out[a * H + b + 1] = g[q][1]; out[(b + 1) * H + a] = g[q][1]; }
        }
    }
}
static int gram_dmma(cudaStream_t st, const Dev& d, const double* X, bool amat, int n, double* out) {
    const int H = d.H, HP8 = (H + 7) & ~7;
    const size_t smem = (size_t)32 * pitch4g(HP8) * sizeof(double);
    const int grid = std::max(1, std::min(cdiv(std::max(n, 1), 32), 148 * (HP8 <= 64 ? 3 : 1)));
#define GD(TP)                                                                                                          \
    if (amat) gram_dmma_kernel<TP, true><<<grid, 256, smem, st>>>(X, n, H, d.ldB, d.part, d.sc);                       \
    else gram_dmma_kernel<TP, false><<<grid, 256, smem, st>>>(X, n, H, d.ldB, d.part, d.sc);
    if (HP8 <= 32) { GD(2) } else if (HP8 <= 64) { GD(5) } else { GD(17) }
#undef GD
    VB_LAUNCH_OK();
    return sum_partials(st, d.part, grid, (size_t)H * H, (size_t)H * H, out, d.sc);
}
static int gram_impl(cudaStream_t st, const Dev& d, const double* X, bool amat, int n, const double* w, int wpow, double* out) {
    const int H = d.H;
    const int nblk = std::max(1, std::min(296, cdiv(std::max(n, 1), 256)));
    const int rpb = cdiv(cdiv(std::max(n, 1), nblk), 32) * 32;
    const size_t smem = (size_t)(32 * (H + 1) + 32) * sizeof(double);
    const int R = cdiv(H, 16);
#define GRAM_LAUNCH(RR)                                                                                              \
    if (amat) gram_partial_kernel<RR, true><<<nblk, 256, smem, st>>>(X, n, H, d.ldB, w, wpow, rpb, d.part, d.sc);     \
    else gram_partial_kernel<RR, false><<<nblk, 256, smem, st>>>(X, n, H, d.ldB, w, wpow, rpb, d.part, d.sc);
    if (R <= 1) { GRAM_LAUNCH(1) } else if (R <= 2) { GRAM_LAUNCH(2) } else if (R <= 4) { GRAM_LAUNCH(4) } else { GRAM_LAUNCH(8) }
#undef GRAM_LAUNCH
    VB_LAUNCH_OK();
    return sum_partials(st, d.part, nblk, (size_t)H * H, (size_t)H * H, out, d.sc);
}
int k_gram(cudaStream_t st, const Dev& d, const double* X, bool amat, int n, const double* w, double* out) {
    if (w == nullptr && n >= 64) return gram_dmma(st, d, X, amat, n, out);     // unweighted: tensor-core path
    return gram_impl(st, d, X, amat, n, w, 1, out);
}
int k_gram_w2(cudaStream_t st, const Dev& d, const double* X, int n, const double* w, double* out) {
    return gram_impl(st, d, X, false, n, w, 2, out);
}

// ------------------------------------------------------------------------------------------- H x H posterior covariances
// mode 0: SigmaA = sigma2*inv(B'B + L*SigmaB + sigma2*invCA)            src/vbmf.jl:96-97
// mode 1: SigmaB = sigma2*inv(A'A + M*SigmaA + sigma2*invCB)            src/vbmf.jl:110-111
// mode 2: SigmaA <- all-reduced sum of per-column blocks; SigmaB = inv(diag(CB) + c*(A'A + SigmaA)),
//         c = sigmaHat or mean(sigmaVecHat)                             src/vbmf_sparse.jl:256-265, src/vbmf_dual.jl:294-303
// Blocked rank-4 Gauss-Jordan on the tensor cores (linalg.cuh::warp_block_gj_sym): a step handles four pivots with one
// barrier and one DMMA per tile.  These inverses sit on the critical path of every iteration, replicated on every GPU.
__device__ __forceinline__ double hxh_elem(const Dev& d, int mode, int diag_var, int i, int j) {
    const Scalars* sc = d.sc;
    const int e = i * d.H + j;
    if (mode == 0) return d.BtB[e] + (double)d.L * d.SigmaB[e] + sc->sigma2 * d.invCA[e];
    if (mode == 1) return (d.packed + packed_ata(d))[e] + (double)d.Mglob * d.SigmaA[e] + sc->sigma2 * d.invCB[e];
    const double c = diag_var ? sc->meanSigmaVec : sc->sigmaHat;
    return ((i == j) ? d.CBv[i] : 0.0) + c * ((d.packed + packed_ata(d))[e] + (d.packed + packed_sa(d))[e]);
}
// H <= 8: one warp, upper-triangular tiles
template <int NT>
__global__ void __launch_bounds__(32, 1) hxh_warp_kernel(Dev d, int mode, int diag_var) {
    ACTIVE_OR_RETURN(d);
    constexpr int NTRI = NT * (NT + 1) / 2;
    __shared__ __align__(16) double scr[GJ_SCRATCH], sv[32];
    const int H = d.H, lane = threadIdx.x, r = lane >> 2, j = lane & 3;
    if (mode == 2) for (int e = lane; e < H * H; e += 32) d.SigmaA[e] = (d.packed + packed_sa(d))[e];
    sv[lane] = lane < H ? rsqrt(hxh_elem(d, mode, diag_var, lane, lane)) : 1.0;
    __syncwarp();
    double c[NTRI][2];
#pragma unroll
    for (int ti = 0; ti < NT; ++ti)
#pragma unroll
        for (int tj = ti; tj < NT; ++tj)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int row = 8 * ti + r, col = 8 * tj + 2 * j + k;
                const double v = (row < H && col < H) ? hxh_elem(d, mode, diag_var, row, col) : (row == col ? 1.0 : 0.0);
                c[tri_idx(ti, tj, NT)][k] = -v * (sv[row] * sv[col]);
            }
    double dummy = 0.0;
    const bool ok = warp_block_gj_sym<NT>(c, dummy, lane, scr);
    if (!ok && lane == 0) d.sc->chol_fail = 1;
    double* out = (mode == 0) ? d.SigmaA : d.SigmaB;
    const double scale = (mode == 2) ? 1.0 : d.sc->sigma2;
    __syncwarp();
#pragma unroll
    for (int ti = 0; ti < NT; ++ti)
#pragma unroll
        for (int tj = ti; tj < NT; ++tj)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int row = 8 * ti + r, col = 8 * tj + 2 * j + k;
                if (row < H && col < H) {
                    const double v = ok ? scale * (c[tri_idx(ti, tj, NT)][k] * (sv[row] * sv[col])) : nan("");
                    out[row * H + col] = v;
                    if (ti != tj) out[col * H + row] = v;
                }
            }
}
// 8 < H <= 128: 16 warps, the full NTD x NTD tile grid spread over the warps (warp w: tile row w / WPR, TPW tile columns).
// Per block step: the owners of the pivot column block publish the panel (double buffered); the first N/32 warps run the
// four sweeps with lane = row (linalg.cuh::gj_panel_sweeps, the 4 x 4 pivot block evolved in every lane) and leave the
// multipliers G and the pre-sweep columns Q in shared memory; every warp then reads its A / B fragments and issues TPW DMMAs.
// Two barriers per four pivots.
template <int NTD, int TPW>
__global__ void __launch_bounds__(512, 1) hxh_dmma_kernel(Dev d, int mode, int diag_var) {
    ACTIVE_OR_RETURN(d);
    constexpr int N = 8 * NTD, WPR = NTD / TPW, PL = N + 4, NRW = N / 32;
    static_assert(NTD * WPR == 16, "16 warps cover the tile grid");
    __shared__ __align__(16) double Ps[2][4 * PL];
    __shared__ __align__(16) double Gs[4 * PL], Qs[4 * PL];
    __shared__ double sv[N];
    __shared__ int s_fail;
    const int H = d.H, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
    const int ti = warp / WPR, tj0 = (warp % WPR) * TPW;
    if (mode == 2) for (int e = threadIdx.x; e < H * H; e += 512) d.SigmaA[e] = (d.packed + packed_sa(d))[e];
    for (int t = threadIdx.x; t < N; t += 512) sv[t] = t < H ? rsqrt(hxh_elem(d, mode, diag_var, t, t)) : 1.0;
    if (threadIdx.x == 0) s_fail = 0;
    __syncthreads();
    const int row = 8 * ti + r;
    double c[TPW][2];                       // T = -(equilibrated matrix), identity padded
#pragma unroll
    for (int u = 0; u < TPW; ++u)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int col = 8 * (tj0 + u) + 2 * j + k;
            const double v = (row < H && col < H) ? hxh_elem(d, mode, diag_var, row, col) : (row == col ? 1.0 : 0.0);
            c[u][k] = -v * (sv[row] * sv[col]);
        }
    const int nsteps = (H + 3) >> 2;
#pragma unroll
    for (int u = 0; u < TPW; ++u)
        if (tj0 + u == 0 && (j >> 1) == 0) { Ps[0][(2 * (j & 1)) * PL + row] = c[u][0]; Ps[0][(2 * (j & 1) + 1) * PL + row] = c[u][1]; }
    for (int s = 0; s < nsteps; ++s) {
        __syncthreads();
        const double* P = Ps[s & 1];
        const int tk = s >> 1, half = s & 1;
        if (warp < NRW) {
            const int rowi = warp * 32 + lane;
            double a[4][4], vk[4] = {0.0, 0.0, 0.0, 0.0}, y[4], gq[4], pq[4], dummy = 0.0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double2 lo = *reinterpret_cast<const double2*>(P + q * PL + 4 * s), hi = *reinterpret_cast<const double2*>(P + q * PL + 4 * s + 2);
                a[0][q] = lo.x; a[1][q] = lo.y; a[2][q] = hi.x; a[3][q] = hi.y;
                y[q] = P[q * PL + rowi];
            }
            if (!gj_panel_sweeps(a, vk, y, dummy, rowi - 4 * s, gq, pq)) s_fail = 1;
#pragma unroll
            for (int q = 0; q < 4; ++q) { Gs[q * PL + rowi] = gq[q]; Qs[q * PL + rowi] = pq[q]; }
        }
        __syncthreads();
        const double wf = Gs[j * PL + row];
#pragma unroll
        for (int u = 0; u < TPW; ++u) dmma884(c[u], wf, Qs[j * PL + 8 * (tj0 + u) + r]);
        if (ti == tk && (r >> 2) == half && j == (r >> 1)) {
#pragma unroll
            for (int u = 0; u < TPW; ++u) if (tj0 + u == tk) { if (r & 1) c[u][1] += 2.0; else c[u][0] += 2.0; }
        }
        if (s + 1 < nsteps) {              // panel of the next step into the other buffer
            const int tkn = (s + 1) >> 1, halfn = (s + 1) & 1;
            double* Pn = Ps[(s + 1) & 1];
#pragma unroll
            for (int u = 0; u < TPW; ++u)
                if (tj0 + u == tkn && (j >> 1) == halfn) { Pn[(2 * (j & 1)) * PL + row] = c[u][0]; Pn[(2 * (j & 1) + 1) * PL + row] = c[u][1]; }
        }
    }
    __syncthreads();
    const bool ok = s_fail == 0;
    if (!ok && threadIdx.x == 0) d.sc->chol_fail = 1;
    double* out = (mode == 0) ? d.SigmaA : d.SigmaB;
    const double scale = (mode == 2) ? 1.0 : d.sc->sigma2;
#pragma unroll
    for (int u = 0; u < TPW; ++u)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int col = 8 * (tj0 + u) + 2 * j + k;
            if (row < H && col < H) out[row * H + col] = ok ? scale * (c[u][k] * (sv[row] * sv[col])) : nan("");
        }
}
static int hxh_launch(cudaStream_t st, const Dev& d, int mode, int dv) {
    const int H = d.H;
    if (H <= 8) hxh_warp_kernel<1><<<1, 32, 0, st>>>(d, mode, dv);
    else if (H <= 32) hxh_dmma_kernel<4, 1><<<1, 512, 0, st>>>(d, mode, dv);   // 16 warps, one tile each: 26 -> ~10 us at H = 32
    else if (H <= 64) hxh_dmma_kernel<8, 4><<<1, 512, 0, st>>>(d, mode, dv);
    else hxh_dmma_kernel<16, 16><<<1, 512, 0, st>>>(d, mode, dv);
    VB_LAUNCH_OK();
    return 0;
}
int k_dense_sigmaA(cudaStream_t st, const Dev& d) { return hxh_launch(st, d, 0, 0); }
int k_sigmaB(cudaStream_t st, const Dev& d, int flags) {
    return hxh_launch(st, d, d.kind == KIND_DENSE ? 1 : 2, (flags & F_DIAG_VAR) ? 1 : 0);
}

// ------------------------------------------------------------------------------------------- dense A epilogue
// AHat = ((Y'*BHat)*SigmaA)/sigma2   src/vbmf.jl:98  (left-to-right association, Q12), label mask (:101), and the Gram
// AHat'AHat that updateB!/updateCA!/updateSigma2! need (src/vbmf.jl:110,131,155) -- one pass over the K1 slabs:
//   T  = sum_s Pslab_s[tile]            (fixed-order split-K reduction, 32 rows x H)
//   An = (T * SigmaA) / sigma2          DMMA, operands in shared memory with row pitch = 4 (mod 16) doubles so that the
//                                       fragment loads (lane (r, j) -> [r][k0+j] resp. [k0+j][r]) hit 16 distinct banks
//   G += An' * An                       DMMA, accumulators live in registers across the CTA's tiles
__device__ __forceinline__ void dmma_acc(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
__host__ __device__ inline int pitch4(int hp8) { return ((hp8 + 11) / 16) * 16 + 4; }

template <int TPW>   // Gram tiles per warp: ceil((HP8/8)^2 / 8)
__global__ void __launch_bounds__(256, (TPW <= 8 ? 3 : 1)) dense_A_fused_kernel(Dev d, const double* __restrict__ slabs, int S, size_t slab_stride,
                                                                                int m_begin, int m_end, int part_base) {
    ACTIVE_OR_RETURN(d);
    extern __shared__ double sm[];
    const int H = d.H, HP8 = (H + 7) & ~7, ld = pitch4(HP8), nt8 = HP8 / 8;
    double* Ss = sm;                 // [HP8][ld]  SigmaA, zero padded
    double* T = Ss + HP8 * ld;       // [32][ld]   P tile
    double* An = T + 32 * ld;        // [32][ld]   new AHat tile
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
    for (int e = threadIdx.x; e < HP8 * ld; e += 256) {
        const int i = e / ld, c = e - i * ld;
        Ss[e] = (i < H && c < H) ? d.SigmaA[i * H + c] : 0.0;
    }
    const double s2 = d.sc->sigma2;
    const int hmask = H - d.H1;      // columns >= hmask are zeroed on labelled rows
    constexpr int NTW = TPW == 2 ? 2 : (TPW == 8 ? 4 : 8);       // column tiles of the product per warp: ceil(nt8 / 2)
    constexpr int GT = TPW == 2 ? 2 : (TPW == 8 ? 5 : 17);       // upper-triangular Gram tiles per warp: ceil(nt8*(nt8+1)/2 / 8)
    double g[GT][2];
    int ga[GT], gb[GT];            // this warp's Gram tiles (at <= bt), -1 = none; idx = warp + 8*q enumerates the upper triangle
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        g[q][0] = 0.0; g[q][1] = 0.0;
        int idx = warp + 8 * q, at = 0;
        while (at < nt8 && idx >= nt8 - at) { idx -= nt8 - at; ++at; }
        ga[q] = at < nt8 ? at : -1;
        gb[q] = at + idx;
    }
    const int ntiles = (m_end - m_begin + 31) / 32;             // rows [m_begin, m_end) of AHat (the whole shard, or one upload chunk)
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int m0 = m_begin + tile * 32, nr = min(32, m_end - m0);
        __syncthreads();
#pragma unroll 4
        for (int e = threadIdx.x; e < 32 * HP8; e += 256) {      // independent loads of several elements in flight
            const int i = e / HP8, c = e - i * HP8;
            double v = 0.0;
            if (i < nr && c < H) {
                const size_t idx = (size_t)(m0 + i) * H + c;
                v = slabs[idx];
                if (S > 1) v += slabs[slab_stride + idx];
                if (S > 2) v += slabs[2 * slab_stride + idx];
                for (int s = 3; s < S; ++s) v += slabs[(size_t)s * slab_stride + idx];
            }
            T[i * ld + c] = v;
        }
        __syncthreads();
        // An = T * SigmaA / sigma2 : warp -> row tile (warp & 3), column tiles (warp >> 2), +2, ... with one independent
        // accumulator per column tile (a single accumulator makes the k loop one dependent chain of DMMAs, 26 clk each)
        {
            const int mt = warp & 3;
            double c2[NTW][2];
#pragma unroll
            for (int u = 0; u < NTW; ++u) { c2[u][0] = 0.0; c2[u][1] = 0.0; }
#pragma unroll 4
            for (int k0 = 0; k0 < HP8; k0 += 4) {
                const double af = T[(8 * mt + r) * ld + k0 + j];
#pragma unroll
                for (int u = 0; u < NTW; ++u) {
                    const int nt = (warp >> 2) + 2 * u;
                    if (nt < nt8) dmma_acc(c2[u], af, Ss[(k0 + j) * ld + 8 * nt + r]);
                }
            }
            const int row = 8 * mt + r;
            const bool lab = d.rowmask != nullptr && row < nr && d.rowmask[m0 + row];
#pragma unroll
            for (int u = 0; u < NTW; ++u) {
                const int nt = (warp >> 2) + 2 * u;
                if (nt < nt8) {
                    const int col = 8 * nt + 2 * j;
                    double v0 = c2[u][0] / s2, v1 = c2[u][1] / s2;
                    if (lab && col >= hmask) v0 = 0.0;
                    if (lab && col + 1 >= hmask) v1 = 0.0;
                    An[row * ld + col] = v0;
                    An[row * ld + col + 1] = v1;
                    if (row < nr) {
                        double* out = d.A + (size_t)(m0 + row) * H + col;
                        if (col < H) out[0] = v0;
                        if (col + 1 < H) out[1] = v1;
                    }
                }
            }
        }
        __syncthreads();
        // G += An' * An over the 32 rows of the tile; G is symmetric, so only the tiles on and above the diagonal are
        // accumulated (tile (bt, at) is the transpose of (at, bt) bit for bit) and mirrored when the partial is written
#pragma unroll
        for (int q = 0; q < GT; ++q) {
            if (ga[q] >= 0) {
#pragma unroll
                for (int i0 = 0; i0 < 32; i0 += 4)
                    dmma_acc(g[q], An[(i0 + j) * ld + 8 * ga[q] + r], An[(i0 + j) * ld + 8 * gb[q] + r]);
            }
        }
    }
    double* out = d.part + (size_t)(part_base + blockIdx.x) * H * H;
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        if (ga[q] >= 0) {
            const int a = 8 * ga[q] + r, b = 8 * gb[q] + 2 * j;
            if (a < H && b < H) { out[a * H + b] = g[q][0]; out[b * H + a] = g[q][0]; }
            if (a < H && b + 1 < H) { out[a * H + b + 1] = g[q][1]; out[(b + 1) * H + a] = g[q][1]; }
        }
    }
}
// slabs: S split-K slabs of K1 (slab_stride apart) or the single P buffer (S = 1); writes AHat rows [m_begin, m_end) and one
// Gram partial per CTA at d.part[(part_base + cta)*H*H]
static int dense_A_fused_launch(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride, int m_begin, int m_end,
                                int part_base, int max_grid, int* grid_out) {
    const int H = d.H, HP8 = (H + 7) & ~7, ld = pitch4(HP8);
    const size_t smem = (size_t)((HP8 + 64) * ld) * sizeof(double);
    const int per_sm = std::max(1, std::min(4, (int)((220 * 1024) / (smem + 1024))));     // latency hiding across CTAs
    const int grid = std::max(1, std::min(std::min(cdiv(m_end - m_begin, 32), 148 * per_sm), max_grid));
    if (HP8 <= 32) dense_A_fused_kernel<2><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, m_begin, m_end, part_base);
    else if (HP8 <= 64) dense_A_fused_kernel<8><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, m_begin, m_end, part_base);
    else dense_A_fused_kernel<32><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, m_begin, m_end, part_base);
    VB_LAUNCH_OK();
    *grid_out = grid;
    return 0;
}
int k_dense_A_fused(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride) {
    if (d.Mloc <= 0) return 0;
    int grid = 0;
    if (dense_A_fused_launch(st, d, slabs, S, slab_stride, 0, d.Mloc, 0, 1 << 30, &grid)) return -1;
    return sum_partials(st, d.part, grid, (size_t)d.H * d.H, (size_t)d.H * d.H, d.packed + packed_ata(d), d.sc);
}
// one column chunk of the shard (first iteration overlapped with the upload of Y): partials land at part_base .. part_base + *nparts
int k_dense_A_fused_range(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride, int m_begin, int m_end,
                          int part_base, int max_parts, int* nparts) {
    *nparts = 0;
    if (m_end <= m_begin) return 0;
    return dense_A_fused_launch(st, d, slabs, S, slab_stride, m_begin, m_end, part_base, max_parts, nparts);
}
// packed.AtA = fixed-order sum of nparts Gram partials in d.part
int k_sum_gram_partials(cudaStream_t st, const Dev& d, int nparts) {
    return sum_partials(st, d.part, nparts, (size_t)d.H * d.H, (size_t)d.H * d.H, d.packed + packed_ata(d), d.sc);
}

// AHat[labels, end-H1+1:end] = 0.0     src/vbmf.jl:101, src/vbmf_sparse.jl:245
__global__ void mask_kernel(Dev d) {
    ACTIVE_OR_RETURN(d);
    const int n = d.nlabels * d.H1;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int li = e / d.H1, c = e - li * d.H1;
        d.A[(size_t)d.labels[li] * d.H + (d.H - d.H1 + c)] = 0.0;
    }
}
int k_mask(cudaStream_t st, const Dev& d) {
    if (d.kind == KIND_DUAL || d.kind == KIND_TRIAL || d.nlabels <= 0 || d.H1 <= 0) return 0;
    const int n = d.nlabels * d.H1;
    mask_kernel<<<std::max(1, std::min(cdiv(n, 256), 592)), 256, 0, st>>>(d);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- sparse / dual A update, diagonal path
// src/vbmf_sparse.jl:204-240 == src/vbmf_dual.jl:244-280.
//   d_h   = sigmaHat*||B[:,h]||^2 + L*SigmaB[h,h]                       (Q3)   [diag_var: sum_l (B[l,h]*sv_l)^2 + L*mean(sv)*SigmaB[h,h], Q4]
//   prec  = [d ; repeat(d, inner = M-1)] + CA                           (Q2: element j>H reads d[ceil((j-H)/(M-1))], global j and M)
//   s     = 1 ./ prec ;  vec(A') = (sigmaHat*s) .* vec(B'Y)             [diag_var: s .* vec(B' diag(sv) Y)]
//   SigmaA = diag(sum_m s[m,:])  -> per-CTA partial column sums, fixed-order reduction into packed.SA
__global__ void __launch_bounds__(256) sparse_A_diag_kernel(Dev d, int diag_var, int rows_per_blk) {
    ACTIVE_OR_RETURN(d);
    __shared__ double dv[128];
    __shared__ double cs[256];
    const int H = d.H;
    const Scalars* sc = d.sc;
    const int nthr = (256 / H) * H;          // every active thread keeps a fixed column h
    for (int h = threadIdx.x; h < H; h += blockDim.x) {
        dv[h] = diag_var ? d.BtBw[h * H + h] + (double)d.L * sc->meanSigmaVec * d.SigmaB[h * H + h]
                         : sc->sigmaHat * d.BtB[h * H + h] + (double)d.L * d.SigmaB[h * H + h];
    }
    __syncthreads();
    const int t = threadIdx.x;
    double colsum = 0.0;
    if (t < nthr) {
        const int m0 = blockIdx.x * rows_per_blk, m1 = min(d.Mloc, m0 + rows_per_blk);
        const double sh = sc->sigmaHat;
        const long long Mg1 = (long long)d.Mglob - 1;
        for (long long e = (long long)m0 * H + t; e < (long long)m1 * H; e += nthr) {
            const long long j0 = (long long)d.moff * H + e;                 // global 0-based index into vec(A')
            const int src = (j0 < H) ? (int)j0 : (int)((j0 - H) / Mg1);
            const double s = 1.0 / (dv[src] + d.CAv[e]);
            const double p = d.P[e];
            d.sdiag[e] = s;
            d.A[e] = diag_var ? s * p : (sh * s) * p;
            colsum += s;
        }
    }
    cs[threadIdx.x] = (t < nthr) ? colsum : 0.0;
    __syncthreads();
    if (t < H) {
        double s = 0.0;
        for (int q = t; q < nthr; q += H) s += cs[q];
        d.part[(size_t)blockIdx.x * H + t] = s;
    }
}
__global__ void __launch_bounds__(256) diag_to_sa_kernel(Dev d, int nparts) {   // packed.SA = diag(sum of partial column sums)
    ACTIVE_OR_RETURN(d);
    const int H = d.H, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* SA = d.packed + packed_sa(d);
    for (int e = threadIdx.x; e < H * H; e += blockDim.x) if (e / H != e % H) SA[e] = 0.0;
    for (int h = warp; h < H; h += 8) {           // one warp per diagonal entry: lane-strided partial sums + fixed shuffle tree
        double s = 0.0;
        for (int p = lane; p < nparts; p += 32) s += d.part[(size_t)p * H + h];
        s = warp_sum(s);
        if (lane == 0) SA[h * H + h] = s;
    }
}
int k_sparse_A_diag(cudaStream_t st, const Dev& d, int flags) {
    const int nblk = std::max(1, std::min(MAX_PARTS, cdiv(std::max(d.Mloc, 1), 64)));
    const int rpb = cdiv(std::max(d.Mloc, 1), nblk);
    sparse_A_diag_kernel<<<nblk, 256, 0, st>>>(d, (flags & F_DIAG_VAR) ? 1 : 0, rpb);
    VB_LAUNCH_OK();
    diag_to_sa_kernel<<<1, 256, 0, st>>>(d, nblk);
    VB_LAUNCH_OK();
    return 0;
}

// Whole-loop version of the diagonal path: ONE pass over vec(A') does what sparse_A_diag + diag_to_sa + mask + update_CA +
// gram_dmma(A) do in five (src/vbmf_sparse.jl:204-246 updateA!, :284-288 updateCA!, src/vbmf_dual.jl:322-351, and the Gram
// AHat'AHat of updateB! :259).  updateCA! only needs this column's a and s and replicated scalars, so hoisting it in front of
// updateB! changes nothing.  Per 32-row tile: P = fixed-order sum of the K1 slabs, s = 1/(d[src] + CA), a = (sigmaHat*s)*P
// (label mask), beta = beta0_g + (a^2 + s)/2, CA = alpha_g/beta; the a tile goes to shared memory for the DMMA Gram
// (accumulators in registers across the CTA's tiles); column sums of s (-> diag SigmaA) and the group sums of the dual /
// trial hyper-prior updates are carried per thread.  Partials per CTA: [H*H Gram | HP8 column sums | 8 group sums].
template <int GT>   // upper-triangular Gram tiles per warp: ceil(nt8*(nt8+1)/2 / 8)
__global__ void __launch_bounds__(256, (GT <= 5 ? 2 : 1)) sparse_A_diag_fused_kernel(Dev d, const double* __restrict__ slabs, int S,
                                                                                    size_t slab_stride, int diag_var) {
    ACTIVE_OR_RETURN(d);
    extern __shared__ double sm[];
    __shared__ double red[32];
    // TR rows per tile.  (128- / 64-row tiles for H <= 32 / 64 -- 16 elements per thread in flight -- measured SLOWER, 106 vs
    // 73 us at 100000 x 32: fewer, longer tiles balance worse over the CTAs; profiles/r02_hbm_kernels_c4_tall_tiles.csv)
    constexpr int TR = 32;
    constexpr int KMAX = GT == 2 ? 4 : (GT == 5 ? 8 : 16);     // elements of a TR x HP8 tile per thread (HP8 <= 32 / 64 / 128)
    __shared__ long long s_q0[TR];
    __shared__ int s_r0[TR];
    const int H = d.H, HP8 = (H + 7) & ~7, ld = pitch4(HP8), nt8 = HP8 / 8;
    double* An = sm;                         // [TR][ld]  new AHat tile (zero padded)
    double* dv = An + TR * ld;               // [HP8]     likelihood part of the diagonal precision
    double* stage = dv + HP8;                // [TR*HP8]  end-of-kernel staging of the per-thread column sums
    Scalars* sc = d.sc;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
    for (int h = threadIdx.x; h < HP8; h += 256) {
        double v = 0.0;
        if (h < H) v = diag_var ? d.BtBw[h * H + h] + (double)d.L * sc->meanSigmaVec * d.SigmaB[h * H + h]
                                : sc->sigmaHat * d.BtB[h * H + h] + (double)d.L * d.SigmaB[h * H + h];
        dv[h] = v;
    }
    const bool grouped = d.kind == KIND_DUAL || d.kind == KIND_TRIAL;
    const double al[3] = {grouped ? sc->alpha00 + 0.5 : sc->alpha, grouped ? sc->alpha01 + 0.5 : sc->alpha, sc->alpha02 + 0.5};
    const double be[3] = {grouped ? sc->beta00 : sc->beta0p, grouped ? sc->beta01 : sc->beta0p, sc->beta02};
    const double sh = sc->sigmaHat;
    const int hmask = H - d.H1;
    const long long Mg1 = (long long)d.Mglob - 1;
    double g[GT][2];
    int gt[GT];
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        g[q][0] = 0.0; g[q][1] = 0.0;
        int idx = warp + 8 * q, at = 0;
        while (at < nt8 && idx >= nt8 - at) { idx -= nt8 - at; ++at; }
        gt[q] = at < nt8 ? (at | ((at + idx) << 8)) : -1;
    }
    double csum[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) csum[k] = 0.0;
    double sca[3] = {0.0, 0.0, 0.0}, slb[3] = {0.0, 0.0, 0.0};
    const int nel = TR * HP8;
    const int ntiles = (d.Mloc + TR - 1) / TR;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int m0 = tile * TR, nr = min(TR, d.Mloc - m0);
        __syncthreads();
        // Q2: element j of vec(A') (0-based, global) reads d[j] for j < H, else d[(j - H) / (M - 1)]: one division per row
        if (threadIdx.x < TR) {
            const long long mg = (long long)d.moff + m0 + threadIdx.x;
            long long q0 = 0; int r0 = 0;
            if (mg > 0 && Mg1 > 0) { const long long base = (mg - 1) * H; q0 = base / Mg1; r0 = (int)(base - q0 * Mg1); }
            s_q0[threadIdx.x] = q0; s_r0[threadIdx.x] = r0;
        }
        __syncthreads();
        // global loads in chunks of KCH elements per thread (independent, many in flight), then the arithmetic of the chunk:
        // one element at a time would serialise ~4 DRAM round trips per element (measured: 1.2 ms at 125000 x 128)
        constexpr int KCH = KMAX < 8 ? KMAX : (GT <= 5 ? 8 : 4);
#pragma unroll
        for (int k0 = 0; k0 < KMAX; k0 += KCH) {
        double pre_p[KCH], pre_ca[KCH];
#pragma unroll
        for (int kk = 0; kk < KCH; ++kk) {
            const int e = threadIdx.x + 256 * (k0 + kk);
            const int i = e / HP8, c = e - i * HP8;
            double p = 0.0, ca = 1.0;
            if (e < nel && i < nr && c < H) {
                const size_t idx = (size_t)(m0 + i) * H + c;
                const double p0 = slabs[idx], p1 = S > 1 ? slabs[slab_stride + idx] : 0.0, p2 = S > 2 ? slabs[2 * slab_stride + idx] : 0.0;
                ca = d.CAv[idx];
                p = p0;
                if (S > 1) p += p1;
                if (S > 2) p += p2;
                for (int s2 = 3; s2 < S; ++s2) p += slabs[(size_t)s2 * slab_stride + idx];
            }
            pre_p[kk] = p; pre_ca[kk] = ca;
        }
#pragma unroll
        for (int kk = 0; kk < KCH; ++kk) {
            const int k = k0 + kk;
            const int e = threadIdx.x + 256 * k;
            if (e < nel) {
                const int i = e / HP8, c = e - i * HP8;
                double a = 0.0;
                if (i < nr && c < H) {
                    const size_t idx = (size_t)(m0 + i) * H + c;
                    const double p = pre_p[kk], ca_in = pre_ca[kk];
                    const long long mg = (long long)d.moff + m0 + i;
                    int src = c;
                    if (mg > 0) {
                        const long long rr = (long long)s_r0[i] + c;
                        src = (int)(s_q0[i] + (rr >= Mg1 ? (Mg1 >= H ? 1 : rr / Mg1) : 0));
                    }
                    const double sv = 1.0 / (dv[src] + ca_in);
                    a = diag_var ? sv * p : (sh * sv) * p;
                    if (d.rowmask != nullptr && c >= hmask && d.rowmask[m0 + i]) a = 0.0;
                    const int grp = (!grouped || c < d.H0) ? 0 : (mg < d.M0 ? 1 : 2);
                    const double beta = (grp == 0 ? be[0] : grp == 1 ? be[1] : be[2]) + 0.5 * (a * a + sv);
                    const double ca = (grp == 0 ? al[0] : grp == 1 ? al[1] : al[2]) / beta;
                    d.sdiag[idx] = sv;
                    d.A[idx] = a;
                    d.beta[idx] = beta;
                    d.CAv[idx] = ca;
                    csum[k] += sv;
                    if (grouped) {
                        const double lb = log(beta);
                        if (grp == 0) { sca[0] += ca; slb[0] += lb; } else if (grp == 1) { sca[1] += ca; slb[1] += lb; } else { sca[2] += ca; slb[2] += lb; }
                    }
                }
                An[i * ld + c] = a;
            }
        }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < GT; ++q) {
            if (gt[q] >= 0) {
                const double* pa = An + j * ld + 8 * (gt[q] & 255) + r;
                const double* pb = An + j * ld + 8 * (gt[q] >> 8) + r;
#pragma unroll 8
                for (int i0 = 0; i0 < TR; i0 += 4) dmma_acc2(g[q], pa[i0 * ld], pb[i0 * ld]);
            }
        }
    }
    const int PS = H * H + HP8 + 8;
    double* out = d.part + (size_t)blockIdx.x * PS;
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        if (gt[q] >= 0) {
            const int a = 8 * (gt[q] & 255) + r, b = 8 * (gt[q] >> 8) + 2 * j;
            if (a < H && b < H) { out[a * H + b] = g[q][0]; out[b * H + a] = g[q][0]; }
            if (a < H && b + 1 < H) { out[a * H + b + 1] = g[q][1]; out[(b + 1) * H + a] = g[q][1]; }
        }
    }
    // column sums of s: element slot (t, k) always holds column (t + 256k) % HP8 -> fixed-order sum over the TR rows of the slot grid
    __syncthreads();
#pragma unroll
    for (int k = 0; k < KMAX; ++k) { const int e = threadIdx.x + 256 * k; if (e < nel) stage[e] = csum[k]; }
    __syncthreads();
    if (threadIdx.x < HP8) {
        double t = 0.0;
        for (int i = 0; i < TR; ++i) t += stage[i * HP8 + threadIdx.x];
        out[H * H + threadIdx.x] = t;
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const double a = block_sum(sca[q], red), b = block_sum(slb[q], red);
        if (threadIdx.x == 0) { out[H * H + HP8 + q] = a; out[H * H + HP8 + 3 + q] = b; }
    }
    if (threadIdx.x == 0) {
        out[H * H + HP8 + 6] = 0.0; out[H * H + HP8 + 7] = 0.0;
        if (blockIdx.x == 0 && grouped) { sc->alpha_g0 = al[0]; sc->alpha_g1 = al[1]; sc->alpha_g2 = al[2]; }
    }
}
// fixed-order reduction of the per-CTA partials: packed.AtA (local Gram), packed.SA = diag(column sums), packed.EX
__global__ void __launch_bounds__(256) sparse_diag_reduce_kernel(Dev d, int nparts) {
    ACTIVE_OR_RETURN(d);
    __shared__ double sm[8][33];
    const int H = d.H, HP8 = (H + 7) & ~7, n = H * H + HP8 + 8;
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int e = blockIdx.x * 32 + x;
    double* SA = d.packed + packed_sa(d);
    for (int q = blockIdx.x * 256 + threadIdx.x; q < H * H; q += gridDim.x * 256) if (q / H != q % H) SA[q] = 0.0;
    double s = 0.0;
    if (e < n) {
#pragma unroll 4
        for (int p = y; p < nparts; p += 8) s += d.part[(size_t)p * n + e];
    }
    sm[y][x] = s;
    __syncthreads();
    if (y == 0 && e < n) {
        double t = sm[0][x];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += sm[k][x];
        if (e < H * H) (d.packed + packed_ata(d))[e] = t;
        else if (e < H * H + HP8) { const int h = e - H * H; if (h < H) SA[h * H + h] = t; }
        else if (d.kind == KIND_DUAL || d.kind == KIND_TRIAL) (d.packed + packed_ex(d))[e - H * H - HP8] = t;
    }
}
static size_t sparse_diag_fused_smem(int H) {
    const int HP8 = (H + 7) & ~7, TR = 32;
    return (size_t)(TR * pitch4(HP8) + HP8 + TR * HP8) * sizeof(double);
}
int k_sparse_diag_reduce(cudaStream_t st, const Dev& d, int nparts) {
    const int H = d.H, HP8 = (H + 7) & ~7;
    sparse_diag_reduce_kernel<<<cdiv(H * H + HP8 + 8, 32), 256, 0, st>>>(d, nparts);
    VB_LAUNCH_OK();
    return 0;
}
// defer_parts != NULL: the fixed-order reduction of the per-CTA partials is left to the caller (k_sparse_diag_reduce on
// another stream: only SigmaB and the tail need its results), *defer_parts = number of partials in d.part
int k_sparse_A_diag_fused(cudaStream_t st, const Dev& d, const double* slabs, int S, size_t slab_stride, int flags, int* defer_parts) {
    const int H = d.H, HP8 = (H + 7) & ~7;
    const int dv = (flags & F_DIAG_VAR) ? 1 : 0;
    const size_t smem = sparse_diag_fused_smem(H);
    const int per_sm = HP8 <= 64 ? 2 : 1, TR = 32;
    const int grid = std::max(1, std::min(cdiv(std::max(d.Mloc, 1), TR), 148 * per_sm));
    if (HP8 <= 32) sparse_A_diag_fused_kernel<2><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, dv);
    else if (HP8 <= 64) sparse_A_diag_fused_kernel<5><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, dv);
    else sparse_A_diag_fused_kernel<17><<<grid, 256, smem, st>>>(d, slabs, S, slab_stride, dv);
    VB_LAUNCH_OK();
    if (defer_parts != nullptr) { *defer_parts = grid; return 0; }
    return k_sparse_diag_reduce(st, d, grid);
}

// ------------------------------------------------------------------------------------------- K4: sparse / dual A update, full covariance
// src/vbmf_sparse.jl:178-202 == src/vbmf_dual.jl:218-242.  inv(sigmaHat*kron(I_M, G0) + diagm(CA)) is block diagonal, so per
// column m:  Sigma_m = inv(G + diag(CA_m)),  G = sigmaHat*(B'B + L*SigmaB)  [diag_var: B'diag(sv)B + L*mean(sv)*SigmaB],
//            a_m = (sigmaHat*Sigma_m)*p_m  [diag_var: Sigma_m*p_m],  diag, SigmaA = sum_m Sigma_m.
// One thread group (warp for H <= 32, CTA otherwise) per matrix, factor held in shared memory.
__global__ void build_G_kernel(Dev d, int diag_var) {
    ACTIVE_OR_RETURN(d);
    const Scalars* sc = d.sc;
    for (int e = threadIdx.x; e < d.H * d.H; e += blockDim.x) {
        d.Gm[e] = diag_var ? d.BtBw[e] + (double)d.L * sc->meanSigmaVec * d.SigmaB[e]
                           : sc->sigmaHat * (d.BtB[e] + (double)d.L * d.SigmaB[e]);
    }
}
template <class G, int QMAX>
__global__ void __launch_bounds__(256) sparse_A_full_kernel(Dev d, int diag_var, int ngroups_total) {
    ACTIVE_OR_RETURN(d);
    extern __shared__ double sm[];
    const int H = d.H, ld = H + 1;
    const Scalars* sc = d.sc;
    G g;
    const int groups_per_cta = blockDim.x / g.size();
    const int gid_in_cta = threadIdx.x / g.size();
    const int gid = blockIdx.x * groups_per_cta + gid_in_cta;
    double* Mx = sm + (size_t)gid_in_cta * (H * ld + 3 * H);
    double* vec = Mx + H * ld;                              // 2H scratch + H for p
    double* pv = vec + 2 * H;
    const double* __restrict__ Gs = d.Gm;                   // H x H, L1/L2 resident
    double acc[QMAX];
#pragma unroll
    for (int q = 0; q < QMAX; ++q) acc[q] = 0.0;
    const int t = g.tid(), n = g.size();
    const double sh = sc->sigmaHat;
    bool all_ok = true;
    for (int m = gid; m < d.Mloc; m += ngroups_total) {
        const double* ca = d.CAv + (size_t)m * H;
        for (int e = t; e < H * H; e += n) {
            const int i = e / H, j = e - i * H;
            Mx[i * ld + j] = Gs[e] + ((i == j) ? ca[i] : 0.0);
        }
        for (int h = t; h < H; h += n) pv[h] = d.P[(size_t)m * H + h];
        g.sync();
        const bool ok = spd_inverse(g, Mx, ld, H, vec);
        all_ok = all_ok && ok;
        for (int h = t; h < H; h += n) {
            double s = 0.0;
            if (diag_var) { for (int k = 0; k < H; ++k) s = fma(Mx[h * ld + k], pv[k], s); }
            else { for (int k = 0; k < H; ++k) s = fma(sh * Mx[h * ld + k], pv[k], s); }
            d.A[(size_t)m * H + h] = ok ? s : nan("");
            d.sdiag[(size_t)m * H + h] = ok ? Mx[h * ld + h] : nan("");
        }
        if (d.blocks != nullptr)
            for (int e = t; e < H * H; e += n) d.blocks[(size_t)m * H * H + e] = Mx[(e / H) * ld + (e % H)];
#pragma unroll
        for (int q = 0; q < QMAX; ++q) {
            const int e = t + q * n;
            if (e < H * H) acc[q] += Mx[(e / H) * ld + (e % H)];
        }
        g.sync();
    }
    if (!all_ok && t == 0) d.sc->chol_fail = 1;
    double* out = d.part + (size_t)gid * H * H;
#pragma unroll
    for (int q = 0; q < QMAX; ++q) {
        const int e = t + q * n;
        if (e < H * H) out[e] = acc[q];
    }
}
// H <= 32: one warp per matrix, upper-triangular 8 x 8 tiles in DMMA accumulator registers, blocked
// rank-4 Gauss-Jordan (linalg.cuh::warp_block_gj_sym).  The right-hand side p_m rides through the sweeps.  The running sum
// of Sigma_m (tiles on and above the diagonal only) lives in registers (ACCS = false) or in per-warp shared memory
// (ACCS = true: 40 registers less, one more CTA per SM).  Shared memory: G as accumulator-layout tiles (read once per matrix
// with conflict-free 128-bit loads), 2.5 KB of scratch per warp.
template <int NT, int MINB, bool ACCS>
__global__ void __launch_bounds__(128, MINB) sparse_A_full_dmma_kernel(Dev d, int diag_var, int nwarps_total) {
    ACTIVE_OR_RETURN(d);
    constexpr int NTRI = NT * (NT + 1) / 2, WPC = 4, SCR = GJ_SCRATCH + 64;
    extern __shared__ __align__(16) double wsm[];
    double* s_G = wsm;                                  // [NTRI][32][2]
    double* s_scr = s_G + NTRI * 64;                    // [WPC][GJ_SCRATCH + 32 + 32]
    double* s_red = s_scr + WPC * SCR;                  // [WPC][NTRI][64] running sums (ACCS) / end-of-kernel reduction
    const int H = d.H;
    const Scalars* sc = d.sc;
    const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5, r = lane >> 2, j = lane & 3;
    const int gw = blockIdx.x * WPC + wic;
    double* scr = s_scr + wic * SCR;
    double* sv = scr + GJ_SCRATCH;                      // [32] equilibration scale 1/sqrt(diag)
    double* cav = sv + 32;                              // [32] CA_m
    double* myred = s_red + wic * NTRI * 64;
    const double sh = sc->sigmaHat;
    const bool live = lane < H;
    // G in accumulator layout, zero padded
    for (int e = threadIdx.x; e < NTRI * 64; e += blockDim.x) {
        const int t = e >> 6, l = (e >> 1) & 31, k = e & 1;
        int ti = 0, rem = t;
        while (rem >= NT - ti) { rem -= NT - ti; ++ti; }
        const int row = 8 * ti + (l >> 2), col = 8 * (ti + rem) + 2 * (l & 3) + k;
        s_G[e] = (row < H && col < H) ? d.Gm[row * H + col] : 0.0;
    }
    const double gll = live ? d.Gm[lane * H + lane] : 0.0;
    double acc[ACCS ? 1 : NTRI][2];
    if (ACCS) {
#pragma unroll
        for (int t = 0; t < NTRI; ++t) *reinterpret_cast<double2*>(myred + t * 64 + lane * 2) = make_double2(0.0, 0.0);
    } else {
#pragma unroll
        for (int t = 0; t < (ACCS ? 1 : NTRI); ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
    }
    __syncthreads();
    bool all_ok = true;
    for (int m = gw; m < d.Mloc; m += nwarps_total) {
        // inputs of column m: CA_m (padded rows / columns: identity) and (Y'B)[m, :].
        // (Fetching them one column ahead with cp.async measured 12 % SLOWER, 0.454 vs 0.407 ms: plain loads stay.)
        double ca = 1.0, p = 0.0;
        if (live) {
            const size_t idx = (size_t)m * H + lane;
            ca = d.CAv[idx];
            p = d.P[idx];
        }
        const double sl = rsqrt(gll + ca);
        sv[lane] = sl;
        cav[lane] = ca;
        __syncwarp();
        double c[NTRI][2];                              // T = -(D*(G + diag(CA_m))*D), D = diag(sl)
        {
            double srow[NT];
            double2 scol[NT];
#pragma unroll
            for (int t = 0; t < NT; ++t) { srow[t] = -sv[8 * t + r]; scol[t] = *reinterpret_cast<const double2*>(sv + 8 * t + 2 * j); }
#pragma unroll
            for (int ti = 0; ti < NT; ++ti)
#pragma unroll
                for (int tj = ti; tj < NT; ++tj) {
                    const int t = tri_idx(ti, tj, NT);
                    const double2 g = *reinterpret_cast<const double2*>(s_G + t * 64 + lane * 2);
                    double g0 = g.x, g1 = g.y;
                    if (ti == tj && j == (r >> 1)) { const double cr = cav[8 * ti + r]; if (r & 1) g1 += cr; else g0 += cr; }
                    c[t][0] = g0 * (srow[ti] * scol[tj].x);
                    c[t][1] = g1 * (srow[ti] * scol[tj].y);
                }
        }
        double v = p * sl;
        const bool ok = warp_block_gj_sym<NT>(c, v, lane, scr);
        all_ok = all_ok && ok;
        const double aval = ok ? (diag_var ? sl * v : (sh * sl) * v) : nan("");
        if (live) d.A[(size_t)m * H + lane] = aval;
        // Sigma_m = D*c*D: un-equilibrate (the scale vector is re-read: holding it across the sweeps costs 24 registers) fused
        // with the running sum; the diagonal (and the blocks on request) are emitted separately
        double srow[NT];
        double2 scol[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) { srow[t] = sv[8 * t + r]; scol[t] = *reinterpret_cast<const double2*>(sv + 8 * t + 2 * j); }
#pragma unroll
        for (int ti = 0; ti < NT; ++ti)
#pragma unroll
            for (int tj = ti; tj < NT; ++tj) {
                const int t = tri_idx(ti, tj, NT);
                const double w0 = srow[ti] * scol[tj].x, w1 = srow[ti] * scol[tj].y;
                if (ACCS) {
                    double2 a = *reinterpret_cast<const double2*>(myred + t * 64 + lane * 2);
                    a.x = fma(c[t][0], w0, a.x); a.y = fma(c[t][1], w1, a.y);
                    *reinterpret_cast<double2*>(myred + t * 64 + lane * 2) = a;
                } else {
                    acc[ACCS ? 0 : t][0] = fma(c[t][0], w0, acc[ACCS ? 0 : t][0]);
                    acc[ACCS ? 0 : t][1] = fma(c[t][1], w1, acc[ACCS ? 0 : t][1]);
                }
                const int row = 8 * ti + r, col = 8 * tj + 2 * j;
                if (ti == tj && j == (r >> 1)) {
                    const double sd = ok ? ((r & 1) ? c[t][1] * w1 : c[t][0] * w0) : nan("");
                    if (row < H) d.sdiag[(size_t)m * H + row] = sd;
                }
                if (d.blocks != nullptr && row < H) {
                    double* blk = d.blocks + (size_t)m * H * H;
                    const double s0 = c[t][0] * w0, s1 = c[t][1] * w1;
                    if (col < H) { blk[row * H + col] = s0; if (ti != tj) blk[col * H + row] = s0; }
                    if (col + 1 < H) { blk[row * H + col + 1] = s1; if (ti != tj) blk[(col + 1) * H + row] = s1; }
                }
            }
        __syncwarp();
    }
    if (!all_ok && lane == 0) d.sc->chol_fail = 1;
    // per-CTA sum of the warps' running sums in fixed warp order; the lower tiles are the mirror image
    if (!ACCS) {
#pragma unroll
        for (int t = 0; t < (ACCS ? 1 : NTRI); ++t) *reinterpret_cast<double2*>(myred + t * 64 + lane * 2) = make_double2(acc[t][0], acc[t][1]);
    }
    __syncthreads();
    double* out = d.part + (size_t)blockIdx.x * H * H;
    for (int e = threadIdx.x; e < H * H; e += blockDim.x) {
        int a = e / H, b = e - a * H;
        if ((a >> 3) > (b >> 3)) { const int tmp = a; a = b; b = tmp; }
        const int t = tri_idx(a >> 3, b >> 3, NT);
        const int idx = t * 64 + (4 * (a & 7) + ((b & 7) >> 1)) * 2 + (b & 1);
        double sum = 0.0;
#pragma unroll
        for (int w = 0; w < WPC; ++w) sum += s_red[w * NTRI * 64 + idx];
        out[e] = sum;
    }
}
template <int NT> static size_t k4_dmma_smem() { return (size_t)(NT * (NT + 1) / 2 * 64 + 4 * (GJ_SCRATCH + 64) + 4 * (NT * (NT + 1) / 2) * 64) * sizeof(double); }

int k_sparse_A_full(cudaStream_t st, const Dev& d, int flags) {
    const int H = d.H;
    const int dv = (flags & F_DIAG_VAR) ? 1 : 0;
    build_G_kernel<<<1, 256, 0, st>>>(d, dv);
    VB_LAUNCH_OK();
    int ngroups;
    if (H <= 32) {
        // CTAs per SM = the instantiation's MINB.  H > 24 keeps the running sums in shared memory for 4 CTAs per SM (measured
        // fastest: 0.407 vs 0.435 ms for 1e5 32 x 32 with 3 CTAs and the sums in registers)
        const int wpc = 4;
        const int per_sm = (H > 16 && H <= 24) ? 3 : 4;
        const int grid = std::max(1, std::min(cdiv(std::max(d.Mloc, 1), wpc), 148 * per_sm));
        ngroups = grid;                                   // one partial per CTA
        if (H <= 8) sparse_A_full_dmma_kernel<1, 4, false><<<grid, 128, k4_dmma_smem<1>(), st>>>(d, dv, grid * wpc);
        else if (H <= 16) sparse_A_full_dmma_kernel<2, 4, false><<<grid, 128, k4_dmma_smem<2>(), st>>>(d, dv, grid * wpc);
        else if (H <= 24) sparse_A_full_dmma_kernel<3, 3, false><<<grid, 128, k4_dmma_smem<3>(), st>>>(d, dv, grid * wpc);
        else sparse_A_full_dmma_kernel<4, 4, true><<<grid, 128, k4_dmma_smem<4>(), st>>>(d, dv, grid * wpc);
    } else {
        const size_t smem = (size_t)(H * (H + 1) + 3 * H) * sizeof(double);
        const int grid = std::max(1, std::min(std::max(d.Mloc, 1), 148));
        ngroups = grid;
        sparse_A_full_kernel<BlockGroup, 64><<<grid, 256, smem, st>>>(d, dv, ngroups);
    }
    VB_LAUNCH_OK();
    return sum_partials(st, d.part, ngroups, (size_t)H * H, (size_t)H * H, d.packed + packed_sa(d), d.sc);
}

// ------------------------------------------------------------------------------------------- element-wise ARD update of vec(A')
// sparse: beta = beta0 + 1/2*(a.^2 + s);  CA = alpha ./ beta                        src/vbmf_sparse.jl:284-288
// dual  : alpha_g = alpha0g + 1/2; beta_g = beta0g + 1/2*(a_g.^2 + s_g); CA_g = alpha_g ./ beta_g, group g = (h > H0)
//         plus the sums the hyper-prior updates need: sum(CA_g), sum(log(beta_g))   src/vbmf_dual.jl:322-351,393-434
__global__ void __launch_bounds__(256) update_CA_kernel(Dev d, int sums_only) {
    ACTIVE_OR_RETURN(d);
    __shared__ double red[32];
    Scalars* sc = d.sc;
    const int H = d.H;
    const bool grouped = d.kind == KIND_DUAL || d.kind == KIND_TRIAL;
    const double al[3] = {grouped ? sc->alpha00 + 0.5 : sc->alpha, grouped ? sc->alpha01 + 0.5 : sc->alpha, sc->alpha02 + 0.5};
    const double be[3] = {grouped ? sc->beta00 : sc->beta0p, grouped ? sc->beta01 : sc->beta0p, sc->beta02};
    double sca[3] = {0.0, 0.0, 0.0}, slb[3] = {0.0, 0.0, 0.0};
    const long long n = (long long)d.Mloc * H;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int h = (int)(e % H);
        const int g = (!grouped || h < d.H0) ? 0 : ((d.moff + (int)(e / H) < d.M0) ? 1 : 2);
        double beta, ca;
        if (sums_only) { beta = d.beta[e]; ca = d.CAv[e]; }      // hyper-prior steps right after an upload: state untouched
        else {
            const double a = d.A[e];
            beta = (g == 0 ? be[0] : g == 1 ? be[1] : be[2]) + 0.5 * (a * a + d.sdiag[e]);
            ca = (g == 0 ? al[0] : g == 1 ? al[1] : al[2]) / beta;
            d.beta[e] = beta;
            d.CAv[e] = ca;
        }
        if (grouped) {
            const double lb = log(beta);
            if (g == 0) { sca[0] += ca; slb[0] += lb; } else if (g == 1) { sca[1] += ca; slb[1] += lb; } else { sca[2] += ca; slb[2] += lb; }
        }
    }
    if (grouped) {
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const double a = block_sum(sca[g], red), b = block_sum(slb[g], red);
            if (threadIdx.x == 0) { d.part[(size_t)blockIdx.x * 8 + g] = a; d.part[(size_t)blockIdx.x * 8 + 3 + g] = b; }
        }
        if (threadIdx.x == 0) {
            d.part[(size_t)blockIdx.x * 8 + 6] = 0.0; d.part[(size_t)blockIdx.x * 8 + 7] = 0.0;
            if (blockIdx.x == 0 && !sums_only) { sc->alpha_g0 = al[0]; sc->alpha_g1 = al[1]; sc->alpha_g2 = al[2]; }
        }
    }
}
int k_update_CA(cudaStream_t st, const Dev& d, int sums_only) {
    const long long n = (long long)d.Mloc * d.H;
    const int grid = std::max(1, (int)std::min<long long>((n + 1023) / 1024, MAX_PARTS));
    update_CA_kernel<<<grid, 256, 0, st>>>(d, sums_only);
    VB_LAUNCH_OK();
    if (d.kind == KIND_DUAL || d.kind == KIND_TRIAL) return sum_partials(st, d.part, grid, 8, 8, d.packed + packed_ex(d), d.sc);
    return 0;
}

int k_sum_slabs(cudaStream_t st, const double* slabs, int S, size_t n, double* out, const Scalars* sc) {
    return sum_partials(st, slabs, S, n, n, out, sc);
}
// fixed-order reduction of the split-K slabs of K2 into the all-reduce payload
int k_reduce_q(cudaStream_t st, const Dev& d, const double* Qpart, int S) {
    const size_t n = (size_t)d.H * d.ldB;
    return sum_partials(st, Qpart, S, n, n, d.packed + packed_q(d), d.sc);
}

// profiling: CTA 0 stamps the phases of its last launch (absolute ns) behind the wait counters
__device__ __forceinline__ void px_stamp(const PxDev& px, int slot) {
    if (px.wait_ns != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
        px.wait_ns[8 + slot] = t;
    }
}
// ---- peer exchange: barrier between the CTAs with the same index b on all ranks.  Slot (b, src) of a rank's flag array is
// written by rank src only and only grows, so `>= epoch` needs no reset.  The release / acquire pair at system scope orders
// this CTA's earlier peer stores (and, through the kernel boundary, everything the stream ran before) ahead of the peers'
// later loads.  A peer that never arrives (a rank that failed on the host) ends the wait after ~30 s with the sticky error
// flag set instead of hanging the device.
__device__ __forceinline__ void px_barrier(const Dev& d, const PxDev& px, int b, unsigned long long ep) {
    __shared__ unsigned long long px_wait_max;
    if (threadIdx.x == 0) px_wait_max = 0;
    __syncthreads();
    if ((int)threadIdx.x < px.W) {
        const int r = threadIdx.x;
        unsigned long long* dst = px.flags[r] + (size_t)b * PX_MAX_WORLD + px.rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(ep) : "memory");
        const unsigned long long* src = px.flags[px.rank] + (size_t)b * PX_MAX_WORLD + r;
        const long long t0 = clock64();
        unsigned long long v, g0 = 0;
        const bool timed = px.wait_ns != nullptr && b == 0;      // profiling: how long CTA 0 waits for its slowest peer
        if (timed) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
            if (v >= ep) break;
            if (clock64() - t0 > 60000000000LL || (*(volatile int*)&d.sc->chol_fail & 4)) { atomicOr(&d.sc->chol_fail, 4); break; }
        }
        if (timed) {
            unsigned long long g1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
            atomicMax(&px_wait_max, g1 - g0);
        }
    }
    __syncthreads();
    if (px.wait_ns != nullptr && b == 0 && threadIdx.x == 0) { atomicAdd(px.wait_ns + 2 * px.site, px_wait_max); atomicAdd(px.wait_ns + 2 * px.site + 1, 1ULL); }
}
// ------------------------------------------------------------------------------------------- B epilogue
__global__ void trbq_kernel(Dev d, int nparts);
// dense : BHat = ((Y*AHat)*SigmaB)/sigma2                       src/vbmf.jl:112
// sparse: BHat = ((sigmaHat*Y)*AHat)*SigmaB                     src/vbmf_sparse.jl:266   (diag_var: diagm(sv)*Y*AHat*SigmaB, :261)
// Fused with everything that needs the new rows while they sit in shared memory: Bold, D = BHat - Bold and the Grams
// BHat'BHat, D'D of the convergence test (src/util.jl:27-29) and of updateCB!/updateSigma*!, and tr(BHat'*(Y*AHat)).
// ---- peer exchange: tile transfers of the row-sharded epilogue.  W is a template parameter and the rounds are real loops so
// that the executed code stays small: a CTA runs this once or twice, and a fully unrolled, predicated 8-rank version spent
// 24-32 us per tile fetching its own instructions (measured: the load phase took that long even with W = 1, all local).
// A 32 x HP8 tile is HP8 * 16 row pairs (16-byte accesses, 256 contiguous bytes per column); two pairs per thread and round.
template <int W>
__device__ __forceinline__ void px_load_tile(const PxDev& px, double* __restrict__ Q, double* __restrict__ T, int ld, int ldB, int l0,
                                             int nr, int H, int HP8, double scale) {
    const int npairs = HP8 * 16;
#pragma unroll 1
    for (int p0 = threadIdx.x; p0 < npairs; p0 += 512) {
        double2 v[2][W];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int p = p0 + 256 * c, h = p >> 4, i = 2 * (p & 15);
            const bool ok = p < npairs && h < H && i < nr;
            const size_t g = (size_t)h * ldB + l0 + i;
#pragma unroll
            for (int rk = 0; rk < W; ++rk) v[c][rk] = ok ? __ldcg(reinterpret_cast<const double2*>(px.packed[rk] + g)) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int p = p0 + 256 * c, h = p >> 4, i = 2 * (p & 15);
            if (p < npairs) {
                double2 q = v[c][0];
#pragma unroll
                for (int rk = 1; rk < W; ++rk) { q.x += v[c][rk].x; q.y += v[c][rk].y; }      // rank order
                if (!(h < H && i < nr)) q = make_double2(0.0, 0.0);
                else {
                    if (i + 1 >= nr) q.y = 0.0;
                    *reinterpret_cast<double2*>(Q + (size_t)h * ldB + l0 + i) = q;      // the row pitch is even: the pad row exists
                }
                T[i * ld + h] = q.x * scale;
                T[(i + 1) * ld + h] = q.y * scale;
            }
        }
    }
}
template <int W>
__device__ __forceinline__ void px_store_tile(const PxDev& px, const double* __restrict__ Bn, int ld, int ldB, int l0, int nr, int H, int HP8) {
    const int npairs = HP8 * 16;
#pragma unroll 1
    for (int p = threadIdx.x; p < npairs; p += 256) {
        const int h = p >> 4, i = 2 * (p & 15);
        if (h < H && i < nr) {
            const double2 b = make_double2(Bn[i * ld + h], Bn[(i + 1) * ld + h]);
            const size_t g = (size_t)h * ldB + l0 + i;
            if (i + 1 < nr) {
#pragma unroll
                for (int rk = 0; rk < W; ++rk) *reinterpret_cast<double2*>(px.B[rk] + g) = b;
            } else {
#pragma unroll
                for (int rk = 0; rk < W; ++rk) px.B[rk][g] = b.x;
            }
        }
    }
}
#define PX_DISPATCH_W(W_, CALL)                                                                  \
    switch (W_) {                                                                                \
        case 1: { constexpr int PW = 1; CALL; } break;                                           \
        case 2: { constexpr int PW = 2; CALL; } break;                                           \
        case 3: { constexpr int PW = 3; CALL; } break;                                           \
        case 4: { constexpr int PW = 4; CALL; } break;                                           \
        case 5: { constexpr int PW = 5; CALL; } break;                                           \
        case 6: { constexpr int PW = 6; CALL; } break;                                           \
        case 7: { constexpr int PW = 7; CALL; } break;                                           \
        default: { constexpr int PW = 8; CALL; } break;                                          \
    }
// DMMA kernel of this epilogue (formulas at the top of the section), for H <= 64 (HP8 = H rounded up to 8, shared pitch = 4 mod 16 as in the A epilogue):
//   Bn = (c .* Qtile) * SigmaB [/ sigma2]        32 x HP8 x HP8 product, 4 x HP8/8 mma tiles over 8 warps
//   G_B += Bn' Bn,  G_D += Dn' Dn                 accumulators in registers across the CTA's tiles
// PX (peer exchange, world > 1): the CTA grid covers only this rank's share of the 32-row tiles; a tile of Q is the sum of
// the peers' local Y*AHat tiles in rank order (the reduce-scatter; the sum is also stored in place, peers never read this
// rank's own rows), and the new BHat rows are written to every peer's BHat (the all-gather).
template <int TPW, bool GRAM, bool PX>   // Gram tiles per warp: ceil((HP8/8)^2 / 8); GRAM = false (H > 64): the Grams come from gram_dmma
__global__ void __launch_bounds__(256, (GRAM ? 2 : 1)) B_epilogue_dmma_kernel(Dev d, int diag_var, PxDev px, int tile_lo, int tile_hi) {
    ACTIVE_OR_RETURN(d);
    extern __shared__ double sm[];
    __shared__ double red[32];
    const int H = d.H, HP8 = (H + 7) & ~7, ld = pitch4(HP8), nt8 = HP8 / 8;
    double* Ss = sm;                 // [HP8][ld] SigmaB, zero padded
    double* T = Ss + HP8 * ld;       // [32][ld]  scaled Q tile
    double* Bn = T + 32 * ld;        // [32][ld]   (GRAM only)
    double* Dn = Bn + 32 * ld;       // [32][ld]   (GRAM only)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
    const Scalars* sc = d.sc;
    double* Q = d.packed + packed_q(d);
    if (PX) px_stamp(px, 0);
    for (int e = threadIdx.x; e < HP8 * ld; e += 256) {
        const int i = e / ld, c = e - i * ld;
        Ss[e] = (i < H && c < H) ? d.SigmaB[i * H + c] : 0.0;
    }
    const bool dense = d.kind == KIND_DENSE;
    const double s2 = sc->sigma2, sh = sc->sigmaHat;
    if (PX) px_stamp(px, 1);
    if (PX) px_barrier(d, px, blockIdx.x, px.epoch + 1);        // every peer's local Y*AHat (split-K reduction) is complete
    if (PX) px_stamp(px, 2);
    constexpr int NTW = TPW == 2 ? 2 : (TPW == 8 ? 4 : 8);      // product column tiles per warp: ceil(nt8 / 2)
    constexpr int GT = GRAM ? (TPW == 2 ? 2 : 5) : 1;           // upper-triangular Gram tiles per warp: ceil(nt8*(nt8+1)/2 / 8)
    double gB[GT][2], gD[GT][2];
    int gt[GT];                                                 // at | bt << 8, -1 = none
#pragma unroll
    for (int q = 0; q < GT; ++q) {
        gB[q][0] = gB[q][1] = 0.0; gD[q][0] = gD[q][1] = 0.0;
        int idx = warp + 8 * q, at = 0;
        while (at < nt8 && idx >= nt8 - at) { idx -= nt8 - at; ++at; }
        gt[q] = at < nt8 ? (at | ((at + idx) << 8)) : -1;
    }
    double tr = 0.0;
    const int ntiles = PX ? tile_hi : (d.L + 31) / 32;
    for (int tile = (PX ? tile_lo : 0) + blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int l0 = tile * 32, nr = min(32, d.L - l0);
        __syncthreads();
        if (PX) {
            const double scale = dense ? 1.0 : sh;
            PX_DISPATCH_W(px.W, px_load_tile<PW>(px, Q, T, ld, d.ldB, l0, nr, H, HP8, scale));
        } else {
            for (int e = threadIdx.x; e < 32 * HP8; e += 256) {
                const int h = e >> 5, i = e & 31;
                double q = 0.0;
                if (i < nr && h < H) {
                    q = Q[(size_t)h * d.ldB + l0 + i];
                    if (!dense) q *= diag_var ? d.sigmaVec[l0 + i] : sh;
                }
                T[i * ld + h] = q;
            }
        }
        __syncthreads();
        if (PX && tile == tile_lo + (int)blockIdx.x) px_stamp(px, 3);       // (the phase stamps describe the CTA's first tile)
        {   // warp -> row tile (warp & 3), column tiles (warp >> 2) + 2u with one independent accumulator each
            const int mt = warp & 3, row = 8 * mt + r;
            double c2[NTW][2];
#pragma unroll
            for (int u = 0; u < NTW; ++u) { c2[u][0] = 0.0; c2[u][1] = 0.0; }
#pragma unroll 4
            for (int k0 = 0; k0 < HP8; k0 += 4) {
                const double af = T[row * ld + k0 + j];
#pragma unroll
                for (int u = 0; u < NTW; ++u) {
                    const int nt = (warp >> 2) + 2 * u;
                    if (nt < nt8) dmma_acc(c2[u], af, Ss[(k0 + j) * ld + 8 * nt + r]);
                }
            }
            // the previous BHat entries first, all in flight together and past L1 (a store to an address whose load is still
            // pending stalls the memory pipe: measured 0.055 -> 0.17 ms at 20000 x 64 when the store followed its load directly)
            double oldv[NTW][2], qv[NTW][2];                  // ... and the Y*AHat entries of tr(BHat' * Y*AHat) with them
#pragma unroll
            for (int u = 0; u < NTW; ++u) {
                const int nt = (warp >> 2) + 2 * u;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int col = 8 * nt + 2 * j + i;
                    const bool ok = nt < nt8 && row < nr && col < H;
                    oldv[u][i] = ok ? __ldcg(d.B + (size_t)col * d.ldB + l0 + row) : 0.0;
                    qv[u][i] = ok ? __ldcg(Q + (size_t)col * d.ldB + l0 + row) : 0.0;
                }
            }
#pragma unroll
            for (int u = 0; u < NTW; ++u) {
                const int nt = (warp >> 2) + 2 * u;
                if (nt < nt8) {
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int col = 8 * nt + 2 * j + i;
                        double bn = 0.0, dn = 0.0;
                        if (row < nr && col < H) {
                            double v = c2[u][i];
                            if (dense) v /= s2;
                            const size_t g = (size_t)col * d.ldB + l0 + row;
                            dn = v - oldv[u][i];
                            if (!GRAM) d.D[g] = dn;              // H > 64: gram_dmma forms D'D from it (with GRAM nobody reads D)
                            if (!PX) d.B[g] = v;                 // PX: all ranks' BHat rows are written from the staged tile below
                            tr = fma(v, qv[u][i], tr);
                            bn = v;
                        }
                        if (GRAM) { Bn[row * ld + col] = bn; Dn[row * ld + col] = dn; }
                    }
                }
            }
        }
        if (GRAM) {
            __syncthreads();
            if (PX) {
                PX_DISPATCH_W(px.W, px_store_tile<PW>(px, Bn, ld, d.ldB, l0, nr, H, HP8));
                if (tile == tile_lo + (int)blockIdx.x) px_stamp(px, 4);
            }
            // symmetric Grams: tiles on and above the diagonal only, mirrored when the partial is written
#pragma unroll
            for (int q = 0; q < GT; ++q) {
                if (gt[q] >= 0) {
                    const int at = gt[q] & 255, bt = gt[q] >> 8;
#pragma unroll
                    for (int i0 = 0; i0 < 32; i0 += 4) {
                        dmma_acc(gB[q], Bn[(i0 + j) * ld + 8 * at + r], Bn[(i0 + j) * ld + 8 * bt + r]);
                        dmma_acc(gD[q], Dn[(i0 + j) * ld + 8 * at + r], Dn[(i0 + j) * ld + 8 * bt + r]);
                    }
                }
            }
        }
    }
    if (PX) px_stamp(px, 5);
    if (GRAM) {
        double* out = d.part + (size_t)blockIdx.x * (2 * H * H + 1);
#pragma unroll
        for (int q = 0; q < GT; ++q) {
            if (gt[q] >= 0) {
                const int a = 8 * (gt[q] & 255) + r, b = 8 * (gt[q] >> 8) + 2 * j;
                if (a < H && b < H) {
                    out[a * H + b] = gB[q][0]; out[b * H + a] = gB[q][0];
                    out[H * H + a * H + b] = gD[q][0]; out[H * H + b * H + a] = gD[q][0];
                }
                if (a < H && b + 1 < H) {
                    out[a * H + b + 1] = gB[q][1]; out[(b + 1) * H + a] = gB[q][1];
                    out[H * H + a * H + b + 1] = gD[q][1]; out[H * H + (b + 1) * H + a] = gD[q][1];
                }
            }
        }
        tr = block_sum(tr, red);
        if (threadIdx.x == 0) out[2 * H * H] = tr;
        if (PX) px_stamp(px, 6);
    } else {
        tr = block_sum(tr, red);
        if (threadIdx.x == 0) d.part[blockIdx.x] = tr;         // Grams follow from gram_dmma on B and D
    }
}
// Global A'A | sum of Sigma blocks | group sums on every rank: the local part goes into this rank's send slot, barrier, sum of
// the peers' slots in rank order, stored in place (peers read the slot, never `packed`).  The slot is rewritten one iteration
// later, behind the Gram-reduction barrier that every peer passes only after it has left this kernel.
__global__ void __launch_bounds__(256) px_small_kernel(Dev d, PxDev px) {
    ACTIVE_OR_RETURN(d);
    const size_t off = packed_ata(d);
    const int n = 2 * d.H * d.H + 8;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e < n) px.small[px.rank][e] = d.packed[off + e];
    px_barrier(d, px, blockIdx.x, px.epoch + 1);
    if (e < n) {
        double v[PX_MAX_WORLD];
#pragma unroll
        for (int rk = 0; rk < PX_MAX_WORLD; ++rk) v[rk] = rk < px.W ? __ldcg(px.small[rk] + e) : 0.0;
        double acc = v[0];
#pragma unroll
        for (int rk = 1; rk < PX_MAX_WORLD; ++rk) if (rk < px.W) acc += v[rk];
        d.packed[off + e] = acc;
    }
}
int k_px_small(cudaStream_t st, const Dev& d, const PxDev& px) {
    const int grid = cdiv(2 * d.H * d.H + 8, 256);
    px_small_kernel<<<grid, 256, 0, st>>>(d, px);
    VB_LAUNCH_OK();
    return 0;
}

// fixed-order reduction of the per-CTA partials: BtB, DtD, sc->trBQ
// PX: the local sum is this rank's partial (its rows of BHat only): it is written to slot `rank` of every peer, and after the
// barrier -- which also says that every peer's BHat rows have landed here -- the rank partials are summed in rank order.
template <bool PX>
__global__ void __launch_bounds__(256) B_reduce_kernel(Dev d, int nparts, PxDev px) {
    ACTIVE_OR_RETURN(d);
    __shared__ double sm[8][33];
    const int H = d.H, n = 2 * H * H + 1;
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int e = blockIdx.x * 32 + x;
    double s = 0.0;
    if (PX) px_stamp(px, 8);
    if (e < n) {
#pragma unroll 4
        for (int p = y; p < nparts; p += 8) s += d.part[(size_t)p * n + e];
    }
    sm[y][x] = s;
    __syncthreads();
    if (PX) px_stamp(px, 9);
    double t = 0.0;
    if (y == 0 && e < n) {
        t = sm[0][x];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += sm[k][x];
    }
    if (PX) {
        if (y == 0 && e < n) {
#pragma unroll
            for (int rk = 0; rk < PX_MAX_WORLD; ++rk) if (rk < px.W) px.gpart[rk][(size_t)px.rank * n + e] = t;
        }
        px_barrier(d, px, blockIdx.x, px.epoch + 1);
        px_stamp(px, 10);
        if (y == 0 && e < n) {
            const double* gp = px.gpart[px.rank];
            t = __ldcg(gp + e);
            for (int rk = 1; rk < px.W; ++rk) t += __ldcg(gp + (size_t)rk * n + e);
        }
    }
    if (y == 0 && e < n) {
        if (e < H * H) d.BtB[e] = t;
        else if (e < 2 * H * H) d.DtD[e - H * H] = t;
        else d.sc->trBQ = t;
    }
    if (PX) px_stamp(px, 11);
}
int k_B_epilogue(cudaStream_t st, const Dev& d, int flags) {
    const int H = d.H, dv = (flags & F_DIAG_VAR) ? 1 : 0;
    if (H <= 64) {
        const int HP8 = (H + 7) & ~7;
        const size_t smem = (size_t)((HP8 + 96) * pitch4(HP8)) * sizeof(double);
        const int grid2 = std::max(1, std::min(cdiv(d.L, 32), 296));      // two CTAs per SM: the tile chain is latency bound
        if (HP8 <= 32) B_epilogue_dmma_kernel<2, true, false><<<grid2, 256, smem, st>>>(d, dv, PxDev(), 0, 0);
        else B_epilogue_dmma_kernel<8, true, false><<<grid2, 256, smem, st>>>(d, dv, PxDev(), 0, 0);
        VB_LAUNCH_OK();
        B_reduce_kernel<false><<<std::max(1, cdiv(2 * H * H + 1, 32)), 256, 0, st>>>(d, grid2, PxDev());
        VB_LAUNCH_OK();
        return 0;
    }
    // H > 64: product-only DMMA epilogue (the Gram accumulators would not fit in registers), Grams by gram_dmma
    const int HP8 = (H + 7) & ~7;
    const size_t smem = (size_t)((HP8 + 32) * pitch4(HP8)) * sizeof(double);
    const int grid3 = std::max(1, std::min(cdiv(d.L, 32), 148));
    B_epilogue_dmma_kernel<1, false, false><<<grid3, 256, smem, st>>>(d, dv, PxDev(), 0, 0);
    VB_LAUNCH_OK();
    trbq_kernel<<<1, 256, 0, st>>>(d, grid3);
    VB_LAUNCH_OK();
    if (gram_dmma(st, d, d.B, false, d.L, d.BtB) || gram_dmma(st, d, d.D, false, d.L, d.DtD)) return -1;
    return 0;
}
// updateB!'s epilogue on this rank's share of the rows (peer exchange, H <= 64, homoscedastic noise)
int k_B_epilogue_px(cudaStream_t st, const Dev& d, int flags, const PxDev& px, int* nparts) {
    const int H = d.H, HP8 = (H + 7) & ~7;
    if (H > 64 || (flags & F_DIAG_VAR)) { set_error("peer-exchange epilogue: H <= 64 and homoscedastic noise only"); return -1; }
    int lo = 0, hi = 0, grid2 = 1;
    px_tile_range(d.L, px.W, px.rank, &lo, &hi, &grid2);
    const size_t smem = (size_t)((HP8 + 96) * pitch4(HP8)) * sizeof(double);
    if (HP8 <= 32) B_epilogue_dmma_kernel<2, true, true><<<grid2, 256, smem, st>>>(d, 0, px, lo, hi);
    else B_epilogue_dmma_kernel<8, true, true><<<grid2, 256, smem, st>>>(d, 0, px, lo, hi);
    VB_LAUNCH_OK();
    *nparts = grid2;
    return 0;
}
int k_B_reduce_px(cudaStream_t st, const Dev& d, const PxDev& px, int nparts) {
    B_reduce_kernel<true><<<std::max(1, cdiv(2 * d.H * d.H + 1, 32)), 256, 0, st>>>(d, nparts, px);
    VB_LAUNCH_OK();
    return 0;
}

__global__ void trbq_kernel(Dev d, int nparts) {
    ACTIVE_OR_RETURN(d);
    __shared__ double red[32];
    double s = 0.0;
    for (int p = threadIdx.x; p < nparts; p += blockDim.x) s += d.part[p];
    s = block_sum(s, red);
    if (threadIdx.x == 0) d.sc->trBQ = s;
}
// tr(BHat' * Q) only (step-level updateSigma / lowerBound when BHat was not just produced by the epilogue)
__global__ void __launch_bounds__(256) trbq_partial_kernel(Dev d) {
    ACTIVE_OR_RETURN(d);
    __shared__ double red[32];
    const double* Q = d.packed + packed_q(d);
    double tr = 0.0;
    const long long n = (long long)d.H * d.ldB;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < n; e += (long long)gridDim.x * 256) {
        const int l = (int)(e % d.ldB);
        if (l < d.L) tr = fma(d.B[e], Q[e], tr);
    }
    tr = block_sum(tr, red);
    if (threadIdx.x == 0) d.part[blockIdx.x] = tr;
}
int k_trbq(cudaStream_t st, const Dev& d) {
    const int grid = std::max(1, std::min(cdiv((long)d.H * d.ldB, 1024), MAX_PARTS));
    trbq_partial_kernel<<<grid, 256, 0, st>>>(d);
    VB_LAUNCH_OK();
    trbq_kernel<<<1, 256, 0, st>>>(d, grid);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- heteroscedastic noise rows
// zetaVec[l] = zeta0 + 1/2*||Y[l,:]||^2 - Y[l,:]*(AHat*BHat[l,:]) + 1/2*traceXTY(A'A + SigmaA, b_l b_l' + SigmaB)
// sigmaVecHat[l] = etaVec[l]/zetaVec[l]                         src/vbmf_sparse.jl:309-316 == src/vbmf_dual.jl:372-379
// Y[l,:]*(AHat*b_l) = Q[l,:]*b_l with Q = Y*AHat already reduced.
__global__ void __launch_bounds__(128) sigma_rows_kernel(Dev d) {
    ACTIVE_OR_RETURN(d);
    extern __shared__ double sm[];
    __shared__ double red[32];
    __shared__ double s_trc;
    const int H = d.H;
    double* GA = sm;   // [H][H]
    const double* AtA = d.packed + packed_ata(d);
    const double* Q = d.packed + packed_q(d);
    double trc = 0.0;
    for (int e = threadIdx.x; e < H * H; e += blockDim.x) {
        const double ga = AtA[e] + d.SigmaA[e];
        GA[e] = ga;
        trc = fma(ga, d.SigmaB[e], trc);
    }
    trc = block_sum(trc, red);
    if (threadIdx.x == 0) s_trc = trc;
    __syncthreads();
    double part = 0.0;
    for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < d.L; l += gridDim.x * blockDim.x) {
        double qb = 0.0, quad = 0.0;
        for (int a = 0; a < H; ++a) {
            const double ba = d.B[(size_t)a * d.ldB + l];
            qb = fma(Q[(size_t)a * d.ldB + l], ba, qb);
            double row = 0.0;
            for (int b = 0; b < H; ++b) row = fma(GA[a * H + b], d.B[(size_t)b * d.ldB + l], row);
            quad = fma(ba, row, quad);
        }
        const double z = d.sc->zeta0 + 0.5 * d.rowY2[l] - qb + 0.5 * (quad + s_trc);
        d.zetaVec[l] = z;
        const double sv = d.etaVec[l] / z;
        d.sigmaVec[l] = sv;
        part += sv;
    }
    part = block_sum(part, red);
    if (threadIdx.x == 0) d.part[blockIdx.x] = part;
}
__global__ void mean_sigma_kernel(Dev d, int nparts) {
    ACTIVE_OR_RETURN(d);
    __shared__ double red[32];
    double s = 0.0;
    for (int p = threadIdx.x; p < nparts; p += blockDim.x) s += d.part[p];
    s = block_sum(s, red);
    if (threadIdx.x == 0) d.sc->meanSigmaVec = s / (double)d.L;
}
int k_sigma_rows(cudaStream_t st, const Dev& d) {
    const int grid = std::max(1, std::min(cdiv(d.L, 128), MAX_PARTS));
    sigma_rows_kernel<<<grid, 128, (size_t)d.H * d.H * 8, st>>>(d);
    VB_LAUNCH_OK();
    mean_sigma_kernel<<<1, 256, 0, st>>>(d, grid);
    VB_LAUNCH_OK();
    return 0;
}
// mean(sigmaVecHat) from the current vector (after an upload)
__global__ void __launch_bounds__(256) mean_only_kernel(Dev d) {
    __shared__ double red[32];
    double s = 0.0;
    for (int l = threadIdx.x; l < d.L; l += blockDim.x) s += d.sigmaVec[l];
    s = block_sum(s, red);
    if (threadIdx.x == 0) d.sc->meanSigmaVec = s / (double)d.L;
}
int k_mean_sigma(cudaStream_t st, const Dev& d) {
    mean_only_kernel<<<1, 256, 0, st>>>(d);
    VB_LAUNCH_OK();
    return 0;
}

// Bs = diag(sigmaVecHat)*BHat : B operand of K1 when diag_var (B' diag(sv) Y, src/vbmf_sparse.jl:193,230)
__global__ void scale_B_kernel(Dev d) {
    ACTIVE_OR_RETURN(d);
    const long long n = (long long)d.H * d.ldB;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int l = (int)(e % d.ldB);
        d.Bs[e] = (l < d.L) ? d.sigmaVec[l] * d.B[e] : 0.0;
    }
}
int k_scale_B(cudaStream_t st, const Dev& d) {
    scale_B_kernel<<<std::max(1, std::min(cdiv((long)d.H * d.ldB, 256), 1184)), 256, 0, st>>>(d);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- post step (single CTA)
// Hyper-parameter / noise updates that only need H x H and scalar data, the convergence test and the loop control.
enum { POST_CA = 1, POST_CB = 2, POST_SIGMA = 4, POST_A00 = 8, POST_A01 = 16, POST_B00 = 32, POST_B01 = 64, POST_DELTA = 128,
       POST_NORM_INIT = 256, POST_A02 = 512, POST_B02 = 1024 };

// inverse digamma on [1e-10, 1e10] by Newton from the left (psi is increasing and concave, so the iteration is monotone);
// stands in for Roots.fzero(f, 1e-10, 1e10) of f(x) = N*log(beta0x) - N*digamma(x) + sum(digamma(alpha) - log(beta_i))
// (src/vbmf_dual.jl:393-401,417-425).  Returns false when there is no sign change in the bracket (Q11: keep the old value).
__device__ bool solve_alpha(double N, double beta0x, double alpha_g, double sum_log_beta, double* root) {
    const double S = N * digamma_pos(alpha_g) - sum_log_beta;      // sum_i gammaELn(alpha_g, beta_i)
    const double c0 = N * log(beta0x);
    const double fa = c0 - N * digamma_pos(1e-10) + S, fb = c0 - N * digamma_pos(1e10) + S;
    if (!isfinite(fa) || !isfinite(fb) || fa * fb > 0.0) return false;
    if (fa == 0.0) { *root = 1e-10; return true; }
    if (fb == 0.0) { *root = 1e10; return true; }
    const double c = (c0 + S) / N;                                  // psi(x) = c
    double x = (c >= -2.22) ? exp(c) + 0.5 : -1.0 / (c + 0.5772156649015329);
    for (int it = 0; it < 100; ++it) {
        const double f = digamma_pos(x) - c;
        double xn = x - f / trigamma_pos(x);
        if (!(xn > 0.0)) xn = 0.5 * x;
        if (fabs(xn - x) <= 2e-16 * fabs(xn)) { x = xn; break; }
        x = xn;
    }
    x = fmin(fmax(x, 1e-10), 1e10);
    *root = x;
    return true;
}

__global__ void __launch_bounds__(256) post_kernel(Dev d, int what, int flags) {
    if (!d.sc->active) return;
    extern __shared__ double sm[];
    __shared__ double red[32];
    Scalars* sc = d.sc;
    const int H = d.H, ld = H + 2;       // even padded size for Jacobi needs ld >= H+1
    double* Mx = sm;                      // [(H+1)][ld]
    double* vec = sm + (H + 2) * ld;      // 4*(H+2)
    const double* AtA = d.packed + packed_ata(d);
    const double* EX = d.packed + packed_ex(d);
    const int t = threadIdx.x;
    BlockGroup g;

    if (d.kind == KIND_DENSE) {
        // updateCA! / updateCB!  src/vbmf.jl:129-146 : C[h,h] = ||X[:,h]||^2/n + Sigma[h,h]; invC = inv(C)
        for (int which = 0; which < 2; ++which) {
            if (!(what & (which == 0 ? POST_CA : POST_CB))) continue;
            double* C = which == 0 ? d.CA : d.CB;
            double* invC = which == 0 ? d.invCA : d.invCB;
            const double* Gm = which == 0 ? AtA : d.BtB;
            const double* Sg = which == 0 ? d.SigmaA : d.SigmaB;
            const double nn = which == 0 ? (double)d.Mglob : (double)d.L;
            __syncthreads();
            for (int h = t; h < H; h += blockDim.x) C[h * H + h] = Gm[h * H + h] / nn + Sg[h * H + h];
            __syncthreads();
            int offdiag = 0;
            for (int e = t; e < H * H; e += blockDim.x) {
                const int i = e / H, j = e - i * H;
                Mx[i * ld + j] = C[e];
                if (i != j && C[e] != 0.0) offdiag = 1;
            }
            offdiag = __syncthreads_or(offdiag);
            if (!offdiag) {
                for (int e = t; e < H * H; e += blockDim.x) {
                    const int i = e / H, j = e - i * H;
                    invC[e] = (i == j) ? 1.0 / C[e] : 0.0;
                }
            } else {
                const bool ok = spd_inverse(g, Mx, ld, H, vec);
                if (!ok && t == 0) sc->chol_fail = 1;
                for (int e = t; e < H * H; e += blockDim.x) invC[e] = ok ? Mx[(e / H) * ld + (e % H)] : nan("");
            }
            __syncthreads();
        }
        if (what & POST_SIGMA) {
            // updateSigma2!  src/vbmf.jl:153-157 ; tr(2*Y'*B*A') = 2*sum(B .* (Y*A)), tr(X*Z) = sum(X .* Z') (symmetric)
            double s = 0.0;
            for (int e = t; e < H * H; e += blockDim.x) {
                const int i = e / H, j = e - i * H;
                const double x = AtA[e] + (double)d.Mglob * d.SigmaA[e];
                const double z = d.BtB[j * H + i] + (double)d.L * d.SigmaB[j * H + i];
                s = fma(x, z, s);
            }
            s = block_sum(s, red);
            if (t == 0) sc->sigma2 = (sc->trYTY - 2.0 * sc->trBQ + s) / ((double)d.L * (double)d.Mglob);
            __syncthreads();
        }
    } else {
        if (what & POST_CB) {
            // updateCB!  src/vbmf_sparse.jl:295-300 (Q6: 1/2*SigmaB[h,h])
            for (int h = t; h < H; h += blockDim.x) {
                const double dl = sc->delta0 + 0.5 * d.BtB[h * H + h] + 0.5 * d.SigmaB[h * H + h];
                d.deltav[h] = dl;
                d.CBv[h] = sc->gamma / dl;
            }
            __syncthreads();
        }
        if ((what & POST_SIGMA) && !(flags & F_DIAG_VAR)) {
            // updateSigma! homoscedastic  src/vbmf_sparse.jl:317-322
            double s = 0.0;
            for (int e = t; e < H * H; e += blockDim.x) {
                const double x = AtA[e] + d.SigmaA[e];
                const double z = d.BtB[e] + (double)d.L * d.SigmaB[e];
                s = fma(x, z, s);
            }
            s = block_sum(s, red);
            if (t == 0) {
                sc->zeta = sc->zeta0 + 0.5 * sc->trYTY - sc->trBQ + 0.5 * s;
                sc->sigmaHat = sc->eta / sc->zeta;
            }
            __syncthreads();
        }
        if ((d.kind == KIND_DUAL || d.kind == KIND_TRIAL) && t == 0) {
            // alphas of every group first, then the betas (they see the new alphas): src/vbmf_dual.jl:491-497,
            // src/vbmf_trial.jl:566-573.  EX = [sum(CA_g) g=0..2 | sum(log(beta_g)) g=0..2]
            const double M1 = (double)d.Mglob - (double)d.M0;
            const double N[3] = {(double)d.Mglob * d.H0, (double)d.M0 * d.H1, M1 * d.H1};
            double r;
            if ((what & POST_A00) && solve_alpha(N[0], sc->beta00, sc->alpha_g0, EX[3], &r)) sc->alpha00 = r;
            if ((what & POST_A01) && solve_alpha(N[1], sc->beta01, sc->alpha_g1, EX[4], &r)) sc->alpha01 = r;
            if ((what & POST_A02) && solve_alpha(N[2], sc->beta02, sc->alpha_g2, EX[5], &r)) sc->alpha02 = r;
            if (what & POST_B00) sc->beta00 = N[0] * sc->alpha00 / EX[0];
            if (what & POST_B01) sc->beta01 = N[1] * sc->alpha01 / EX[1];
            if (what & POST_B02) sc->beta02 = N[2] * sc->alpha02 / EX[2];
        }
        __syncthreads();
    }

    if (what & (POST_DELTA | POST_NORM_INIT)) {
        // delta(new, old) = norm(old - new)/norm(old), src/util.jl:27-29; the two norms come from norms_kernel
        if (t == 0) {
            if (what & POST_DELTA) {
                const double dd = sc->normD / sc->normBold;
                sc->d = dd;
                sc->iter += 1;
                sc->active = (sc->iter < sc->niter) && (dd > sc->eps) ? 1 : 0;
            }
            sc->normBold = sc->normBnew;
        }
    }
}
// norm(BHat - Bold) (block 0) and norm(BHat) (block 1) from the Grams D'D, B'B: Julia 0.5 norm(::Matrix) = sigma_max (Q1)
// = sqrt(lambda_max(Gram)); frobenius mode = sqrt(trace).
__global__ void __launch_bounds__(512) norms_kernel(Dev d, int first) {
    if (!d.sc->active) return;
    extern __shared__ double sm[];
    __shared__ double red[32];
    Scalars* sc = d.sc;
    const int H = d.H, ld = H + 1, t = threadIdx.x;
    const int which = first + blockIdx.x;            // 0: D'D   1: B'B
    const double* Gm = which == 0 ? d.DtD : d.BtB;
    double* Mx = sm;
    double* vec = sm + H * ld;
    double val;
    if (sc->norm_mode == 1) {
        double s = 0.0;
        for (int h = t; h < H; h += blockDim.x) s += Gm[h * H + h];
        val = block_sum(s, red);
    } else {
        for (int e = t; e < H * H; e += blockDim.x) {
            const int i = e / H, j = e - i * H;
            Mx[i * ld + j] = 0.5 * (Gm[i * H + j] + Gm[j * H + i]);
        }
        __syncthreads();
        val = sym_lambda_max(Mx, ld, H, vec);
    }
    if (t == 0) {
        const double nv = sqrt(fmax(val, 0.0)) + (val != val ? val : 0.0);
        if (which == 0) sc->normD = nv; else sc->normBnew = nv;
    }
}
static size_t post_smem(int H) { return (size_t)((H + 2) * (H + 2) + 4 * (H + 2) + 8) * sizeof(double); }
static int post_launch(cudaStream_t st, const Dev& d, int what, int flags) {
    if (what & (POST_DELTA | POST_NORM_INIT)) {
        const int first = (what & POST_DELTA) ? 0 : 1;
        norms_kernel<<<2 - first, 512, post_smem(d.H), st>>>(d, first);
        VB_LAUNCH_OK();
    }
    post_kernel<<<1, 256, post_smem(d.H), st>>>(d, what, flags);
    VB_LAUNCH_OK();
    return 0;
}
int k_post(cudaStream_t st, const Dev& d, int flags, bool with_delta) {
    int what = with_delta ? POST_DELTA : 0;
    if (d.kind == KIND_DENSE) {
        if (flags & F_EST_COVS) what |= POST_CA | POST_CB;
        if (flags & F_EST_VAR) what |= POST_SIGMA;
    } else {
        if (flags & F_EST_CB) what |= POST_CB;
        what |= POST_SIGMA;
        if (d.kind == KIND_DUAL && (flags & F_EST_PRIORS)) what |= POST_A00 | POST_A01 | POST_B00 | POST_B01;
        if (d.kind == KIND_TRIAL && (flags & F_EST_PRIORS)) what |= POST_A00 | POST_A01 | POST_A02 | POST_B00 | POST_B01 | POST_B02;
    }
    return post_launch(st, d, what, flags);
}
int k_norms_init(cudaStream_t st, const Dev& d) { return post_launch(st, d, POST_NORM_INIT, 0); }
int k_updateCB_only(cudaStream_t st, const Dev& d) { return post_launch(st, d, POST_CB, 0); }
int k_dense_cov_only(cudaStream_t st, const Dev& d, int which) { return post_launch(st, d, which == 0 ? POST_CA : POST_CB, 0); }
int k_sigma_only(cudaStream_t st, const Dev& d, int flags) { return post_launch(st, d, POST_SIGMA, flags); }
int k_prior_only(cudaStream_t st, const Dev& d, int which) {
    static const int bits[6] = {POST_A00, POST_A01, POST_A02, POST_B00, POST_B01, POST_B02};
    return post_launch(st, d, bits[which], 0);
}

// ------------------------------------------------------------------------------------------- K10: YHat = BHat*AHat'
// src/vbmf.jl:120-122, src/vbmf_sparse.jl:275-277 -- on demand only (L x M output).
__global__ void __launch_bounds__(256) yhat_kernel(Dev d, double* __restrict__ out, int ldo) {
    extern __shared__ double sm[];
    const int H = d.H;
    double* Bt = sm;            // [64][H+1]
    double* At = sm + 64 * (H + 1);   // [16][H]
    const int l0 = blockIdx.x * 64, m0 = blockIdx.y * 16;
    for (int e = threadIdx.x; e < 64 * H; e += 256) {
        const int h = e >> 6, i = e & 63;
        Bt[i * (H + 1) + h] = (l0 + i < d.L) ? d.B[(size_t)h * d.ldB + l0 + i] : 0.0;
    }
    for (int e = threadIdx.x; e < 16 * H; e += 256) {
        const int r = e / H;
        At[e] = (m0 + r < d.Mloc) ? d.A[(size_t)(m0 + r) * H + (e - r * H)] : 0.0;
    }
    __syncthreads();
    const int i = threadIdx.x & 63, c0 = threadIdx.x >> 6;
    for (int c = c0; c < 16; c += 4) {
        double s = 0.0;
        for (int h = 0; h < H; ++h) s = fma(Bt[i * (H + 1) + h], At[c * H + h], s);
        if (l0 + i < d.L && m0 + c < d.Mloc) out[(size_t)(m0 + c) * ldo + l0 + i] = s;
    }
}
int k_yhat(cudaStream_t st, const Dev& d, double* out, int ldo) {
    if (d.L <= 0 || d.Mloc <= 0) return 0;
    dim3 grid(cdiv(d.L, 64), cdiv(d.Mloc, 16));
    yhat_kernel<<<grid, 256, (size_t)(64 * (d.H + 1) + 16 * d.H) * 8, st>>>(d, out, ldo);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- K7: lower bound
// lowerBound / lowerBoundTrimmed: src/vbmf_sparse.jl:435-489, src/vbmf_dual.jl:556-617.  Phase 0 streams the local slice of
// the MH-length vectors into 9 sums (fixed-order), phase 1 (after the cross-shard all-reduce) assembles the scalar.
//   acc[0..2] sum(log(beta_g)) all elements, group 0..2      acc[3..5] sum(CA_g) all elements
//   acc[6] sum(log(beta)) kept   acc[7] sum(CA) kept   acc[8] sum(CA.*(a.^2+s)) kept   acc[9] sum(log(s)) kept   acc[10] #kept
__global__ void __launch_bounds__(256) lb_partial_kernel(Dev d, double trim, int trimmed) {
    __shared__ double red[32];
    const int H = d.H;
    const bool grouped = d.kind == KIND_DUAL || d.kind == KIND_TRIAL;
    double a[11];
#pragma unroll
    for (int i = 0; i < 11; ++i) a[i] = 0.0;
    const long long n = (long long)d.Mloc * H;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int h = (int)(e % H);
        const int g = (!grouped || h < d.H0) ? 0 : ((d.moff + (int)(e / H) < d.M0) ? 1 : 2);
        lb_accumulate(a, g, d.A[e], d.beta[e], d.CAv[e], d.sdiag[e], trim, trimmed);
    }
#pragma unroll
    for (int i = 0; i < 11; ++i) {
        const double v = block_sum(a[i], red);
        if (threadIdx.x == 0) d.part[(size_t)blockIdx.x * 11 + i] = v;
    }
}
__global__ void lb_reduce_kernel(Dev d, int nparts) {
    const int i = threadIdx.x;
    if (i < 11) {
        double s = 0.0;
        for (int p = 0; p < nparts; ++p) s += d.part[(size_t)p * 11 + i];
        d.lbacc[i] = s;
    }
}

__global__ void lb_final_kernel(Dev d, int trimmed) {
    extern __shared__ double W[];
    if (threadIdx.x != 0) return;
    const int H = d.H;
    const double L = d.L;
    const double* AtA = d.packed + packed_ata(d);
    double tGAGB = 0.0, trCBGB = 0.0, sumCB = 0.0, sumLogDelta = 0.0;
    for (int e = 0; e < H * H; ++e) tGAGB = fma(AtA[e] + d.SigmaA[e], d.BtB[e] + L * d.SigmaB[e], tGAGB);
    for (int h = 0; h < H; ++h) {
        trCBGB = fma(d.CBv[h], d.BtB[h * H + h] + L * d.SigmaB[h * H + h], trCBGB);
        sumCB += d.CBv[h];
        sumLogDelta += log(d.deltav[h]);
    }
    LbInputs in;
    in.kind = d.kind; in.H = H; in.H0 = d.H0; in.H1 = d.H1;
    in.L = L; in.M = d.Mglob; in.M0 = (double)d.M0;
    in.acc = d.lbacc;
    in.tGAGB = tGAGB; in.trCBGB = trCBGB; in.sumCB = sumCB; in.sumLogDelta = sumLogDelta; in.trBQ = d.sc->trBQ;
    in.entropyB = normal_entropy_kron<false>(d.SigmaB, H, d.L, W, nullptr);
    d.sc->lb = lb_assemble(d.sc, in);
}
int k_lower_bound(cudaStream_t st, const Dev& d, double trim, int trimmed, int phase) {
    if (phase == 0) {
        const long long n = (long long)d.Mloc * d.H;
        const int grid = std::max(1, (int)std::min<long long>((n + 1023) / 1024, MAX_PARTS));
        lb_partial_kernel<<<grid, 256, 0, st>>>(d, trim, trimmed);
        VB_LAUNCH_OK();
        lb_reduce_kernel<<<1, 32, 0, st>>>(d, grid);
        VB_LAUNCH_OK();
    } else {
        lb_final_kernel<<<1, 32, (size_t)d.H * d.H * 8, st>>>(d, trimmed);
        VB_LAUNCH_OK();
    }
    return 0;
}

// ------------------------------------------------------------------------------------------- K9: synthetic inputs
// Philox4x32-10 counter-based normals; the stream of Y[:, m] depends only on (seed, global column m), so any sharding of
// the columns generates the same matrix (SURVEY 8(d)).
__device__ __forceinline__ void philox4x32(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ double philox_normal(uint64_t seed, uint64_t stream, uint64_t idx) {
    uint32_t c[4] = {(uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
    philox4x32(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint64_t a = ((uint64_t)c[0] << 32) | c[1], b = ((uint64_t)c[2] << 32) | c[3];
    const double u1 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}
__global__ void randn_kernel(double* x, size_t n, uint64_t seed, uint64_t stream, uint64_t offset) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        x[i] = philox_normal(seed, stream, offset + i);
}
int k_randn(cudaStream_t st, double* x, size_t n, uint64_t seed, uint64_t stream) {
    if (n == 0) return 0;
    randn_kernel<<<std::max(1, std::min(cdiv((long)n, 256), 2368)), 256, 0, st>>>(x, n, seed, stream, 0);
    VB_LAUNCH_OK();
    return 0;
}
// Y[l, m] = sum_r B0[l, r]*A0[mg, r] + noise*E[l, mg],  B0 ~ stream 1, A0 ~ stream 2, E ~ stream 3 (mg = global column)
__global__ void __launch_bounds__(256) synth_kernel(double* __restrict__ Y, int ldY, int L, int Mloc, int moff, int rank,
                                                    double noise, uint64_t seed) {
    extern __shared__ double sm[];
    double* B0 = sm;                 // [64][rank]
    double* A0 = sm + 64 * rank;     // [16][rank]
    const int l0 = blockIdx.x * 64, m0 = blockIdx.y * 16;
    for (int e = threadIdx.x; e < 64 * rank; e += 256)
        B0[e] = philox_normal(seed, 1, (uint64_t)(l0 + e / rank) * rank + (e % rank));
    for (int e = threadIdx.x; e < 16 * rank; e += 256)
        A0[e] = philox_normal(seed, 2, (uint64_t)(moff + m0 + e / rank) * rank + (e % rank));
    __syncthreads();
    const int i = threadIdx.x & 63;
    for (int c = threadIdx.x >> 6; c < 16; c += 4) {
        const int l = l0 + i, m = m0 + c;
        if (l < L && m < Mloc) {
            double s = 0.0;
            for (int r = 0; r < rank; ++r) s = fma(B0[i * rank + r], A0[c * rank + r], s);
            s += noise * philox_normal(seed, 3, (uint64_t)(moff + m) * (uint64_t)L + l);
            Y[(size_t)m * ldY + l] = s;
        }
    }
}
int k_synth(cudaStream_t st, double* Y, int ldY, int L, int Mloc, int moff, int rank, double noise, uint64_t seed) {
    if (L <= 0 || Mloc <= 0) return 0;
    if (rank > 256) { set_error("synthetic rank %d > 256", rank); return -1; }
    dim3 grid(cdiv(L, 64), cdiv(Mloc, 16));
    synth_kernel<<<grid, 256, (size_t)80 * rank * 8, st>>>(Y, ldY, L, Mloc, moff, rank, noise, seed);
    VB_LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------------- per-device kernel attributes
// cudaFuncSetAttribute applies to the CURRENT device only, so every context opts the kernels of this file into their dynamic
// shared memory once for its own device (a process may hold contexts on several GPUs).
#define VB_SMEM_ATTR(kernel, bytes) VB_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)))
int kernels_init_device() {
    const int mxA = (int)((128 + 64) * pitch4(128) * 8);
    VB_SMEM_ATTR(dense_A_fused_kernel<2>, mxA);
    VB_SMEM_ATTR(dense_A_fused_kernel<8>, mxA);
    VB_SMEM_ATTR(dense_A_fused_kernel<32>, mxA);
    VB_SMEM_ATTR(sparse_A_diag_fused_kernel<2>, sparse_diag_fused_smem(32));
    VB_SMEM_ATTR(sparse_A_diag_fused_kernel<5>, sparse_diag_fused_smem(64));
    VB_SMEM_ATTR(sparse_A_diag_fused_kernel<17>, sparse_diag_fused_smem(128));
    VB_SMEM_ATTR((sparse_A_full_kernel<BlockGroup, 64>), (128 * 129 + 384) * 8);
    VB_SMEM_ATTR((sparse_A_full_dmma_kernel<1, 4, false>), k4_dmma_smem<1>());
    VB_SMEM_ATTR((sparse_A_full_dmma_kernel<2, 4, false>), k4_dmma_smem<2>());
    VB_SMEM_ATTR((sparse_A_full_dmma_kernel<3, 3, false>), k4_dmma_smem<3>());
    VB_SMEM_ATTR((sparse_A_full_dmma_kernel<4, 4, true>), k4_dmma_smem<4>());
    const int mxB = (int)((64 + 96) * pitch4(64) * 8);
    VB_SMEM_ATTR((B_epilogue_dmma_kernel<2, true, false>), mxB);
    VB_SMEM_ATTR((B_epilogue_dmma_kernel<8, true, false>), mxB);
    VB_SMEM_ATTR((B_epilogue_dmma_kernel<2, true, true>), mxB);
    VB_SMEM_ATTR((B_epilogue_dmma_kernel<8, true, true>), mxB);
    VB_SMEM_ATTR((B_epilogue_dmma_kernel<1, false, false>), (128 + 32) * pitch4(128) * 8);
    VB_SMEM_ATTR(sigma_rows_kernel, 128 * 128 * 8);
    VB_SMEM_ATTR(post_kernel, post_smem(128));
    VB_SMEM_ATTR(norms_kernel, post_smem(128));
    VB_SMEM_ATTR(yhat_kernel, (64 * 129 + 16 * 128) * 8);
    VB_SMEM_ATTR(lb_final_kernel, 128 * 128 * 8);
    return 0;
}

}  // namespace vb
