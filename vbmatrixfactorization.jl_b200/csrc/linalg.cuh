// Small dense linear algebra on shared memory, cooperative over a thread group (a warp or a whole CTA):
//   * SPD inverse by diagonal equilibration + Cholesky (replaces Julia `inv` = LU getrf/getri on the H x H posterior
//     precision matrices: src/vbmf.jl:96,110,133,145; src/vbmf_sparse.jl:188,259,265; src/vbmf_dual.jl:228,297,303).
//     ARD pruning drives prior precisions to ~1e10 next to O(1) entries (seen in the reference's own log), so the
//     matrix is symmetrically scaled to unit diagonal before factorising.
//   * largest eigenvalue of a symmetric PSD matrix by parallel-order cyclic Jacobi (for Julia 0.5 `norm(::Matrix)`
//     = spectral norm in `delta`, src/util.jl:27-29).
#pragma once
#include "common.cuh"

namespace vb {

struct BlockGroup {
    __device__ __forceinline__ int tid() const { return threadIdx.x; }
    __device__ __forceinline__ int size() const { return blockDim.x; }
    __device__ __forceinline__ void sync() const { __syncthreads(); }
};
struct WarpGroup {
    __device__ __forceinline__ int tid() const { return threadIdx.x & 31; }
    __device__ __forceinline__ int size() const { return 32; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};

// In-place inverse of the SPD matrix A (H x H, row stride ld, shared memory).  `vec` = 2*H doubles of scratch.
// Diagonal equilibration to unit diagonal, then H symmetric Gauss-Jordan sweeps without pivoting (every pivot of an SPD
// matrix is positive; elimination on the equilibrated matrix is as accurate as Cholesky up to a modest constant), two
// group barriers per sweep.  Returns false (for every thread of the group) when a pivot is not positive / not finite.
template <class G>
__device__ bool spd_inverse(const G& g, double* A, int ld, int H, double* vec) {
    const int t = g.tid(), n = g.size();
    double* scal = vec;
    double* col = vec + H;
    bool ok = true;
    for (int i = t; i < H; i += n) scal[i] = 1.0 / sqrt(A[i * ld + i]);
    g.sync();
    for (int e = t; e < H * H; e += n) {
        const int i = e / H, j = e - i * H;
        A[i * ld + j] *= scal[i] * scal[j];
    }
    g.sync();
    for (int k = 0; k < H; ++k) {
        // sweep on pivot k:  A <- [[ A11 - a a'/d , a/d ], [ a'/d , -1/d ]] (sign fixed at the end), a = column k
        const double d = A[k * ld + k];
        if (!(d > 0.0) || !(d < 1e300)) ok = false;
        const double id = 1.0 / d;
        for (int i = t; i < H; i += n) col[i] = A[i * ld + k];
        g.sync();
        for (int e = t; e < H * H; e += n) {
            const int i = e / H, j = e - i * H;
            double v;
            if (i == k) v = (j == k) ? -id : col[j] * id;
            else if (j == k) v = col[i] * id;
            else v = A[i * ld + j] - col[i] * col[j] * id;
            A[i * ld + j] = v;
        }
        g.sync();
    }
    // after sweeping every pivot A holds -inv; undo the sign and the scaling
    for (int e = t; e < H * H; e += n) {
        const int i = e / H, j = e - i * H;
        A[i * ld + j] = -A[i * ld + j] * scal[i] * scal[j];
    }
    g.sync();
    return ok;
}

// ---------------------------------------------------------------------------------------------------------------------
// Register-resident variants of the same equilibrated Gauss-Jordan inverse (the matrix never lives in shared memory).
//
// Warp version, H <= HP <= 32 (HP compile time so every register index is static): lane l owns column l, a[q] = A[q][l].
// In sweep k every lane already holds A[k][l] (= A[l][k]) in a[k]; the lanes publish that row through a 32-double shared
// vector (one STS) and read the whole column back as broadcasts (LDS.128), so a sweep costs ~2 FP64 ops per element and one
// __syncwarp.  Rows / lanes >= H must be padded with the identity by the caller.  col = 64 doubles per warp (double buffer).
// `dg` = A[l][l] of this lane.  On return a[q] = inv(A)[q][l]; `ok` is uniform across the warp.
template <int HP>
__device__ __forceinline__ bool warp_spd_inverse_reg(double (&a)[HP], double dg, int lane, double* col) {
    bool ok = true;
    const double sl = 1.0 / sqrt(dg);
    col[lane] = sl;
    __syncwarp();
#pragma unroll
    for (int q = 0; q < HP; q += 2) {
        const double2 sq = *reinterpret_cast<const double2*>(col + q);
        a[q] *= sq.x * sl;
        a[q + 1] *= sq.y * sl;
    }
    // Software-pipelined sweeps: row k+1 is final as soon as its one FMA of sweep k is done, so it is updated FIRST and
    // published for the next sweep while the other HP-1 FMAs of sweep k still issue; the shared-memory round trip and
    // the reciprocal of the next pivot then overlap with them instead of heading every sweep's dependency chain.
    col[32 + lane] = a[0];
    __syncwarp();
#pragma unroll
    for (int k = 0; k < HP; ++k) {
        const double* c = col + ((k + 1) & 1) * 32;            // row k == column k (symmetry), published by sweep k-1
        double* cn = col + (k & 1) * 32;                       // row k+1 goes here
        const double myk = a[k];                               // A[k][l]
        const double d = c[k];
        if (!(d > 0.0) || !(d < 1e300)) ok = false;
        const double id = 1.0 / d;
        const double t = myk * id;
        const bool piv = lane == k;
        // one FMA per element for every lane: the pivot lane's own column IS column k (a[q] == ck), so
        // ck*(id - 1) + a[q] = ck*id there; elsewhere a[q] - ck*t
        const double beta = piv ? id - 1.0 : -t;
        if (k + 1 < HP) {
            a[k + 1] = fma(c[k + 1], beta, a[k + 1]);
            cn[lane] = a[k + 1];
        }
#pragma unroll
        for (int q = 0; q < HP; q += 2) {
            const double2 ck = *reinterpret_cast<const double2*>(c + q);
            if (q != k + 1) a[q] = fma(ck.x, beta, a[q]);
            if (q + 1 != k + 1) a[q + 1] = fma(ck.y, beta, a[q + 1]);
        }
        a[k] = piv ? -id : t;
        __syncwarp();
    }
    __syncwarp();
    col[lane] = sl;
    __syncwarp();
#pragma unroll
    for (int q = 0; q < HP; q += 2) {
        const double2 sq = *reinterpret_cast<const double2*>(col + q);
        a[q] = -a[q] * sq.x * sl;
        a[q + 1] = -a[q + 1] * sq.y * sl;
    }
    __syncwarp();
    return ok;
}

// ---------------------------------------------------------------------------------------------------------------------
// Blocked (rank-4) symmetric Gauss-Jordan on FP64 tensor-core fragments: the inverse the per-column full-covariance update
// needs 1e5 times per iteration (src/vbmf_sparse.jl:188, src/vbmf_dual.jl:228) and the H x H posterior covariances.
//
// One warp holds T = -S, S an equilibrated SPD matrix of order N = 8*NT (NT <= 4), as the upper-triangular 8 x 8 tiles
// (ti <= tj) of the DMMA accumulator layout: lane = 4*r + j holds T[8ti + r][8tj + 2j], T[8ti + r][8tj + 2j + 1].  A block step
// sweeps the four pivots K = 4s .. 4s+3 at once:
//   1. the column panel Y0 = T[:, K] (N x 4) and the right-hand side go to shared memory (tiles below the diagonal are read
//      through symmetry);
//   2. with lane = row, every lane runs the four sweeps on its own panel row.  The current pivot row of each sweep is not
//      communicated: every lane reads the 4 x 4 pivot block once and evolves it in registers alongside (24 FMAs);
//   3. the update of every stored tile is ONE DMMA.8x8x4 assembled from the sweeps' own terms,
//          T[ti][tj] += G[ti] * Q[tj]^T,   G[:, c] = multipliers of sweep c,   Q[:, c] = column c right before its sweep,
//      (+1 on the pivot entry of Q, so the same product also writes the swept pivot rows / columns; +2 on the block's diagonal).
//      Using the FINISHED panel times the ORIGINAL panel instead (X*inv(D)*X') is algebraically the same update but loses
//      accuracy like the condition number of the 4 x 4 pivot block -- measured: 1e-7 instead of 2e-11 on A = P*Sigma at
//      kappa = 8e4 (tools/k4bench/acc_variants.py); the sequential terms reproduce the rank-1 sweep's rounding behaviour.
// Keeping -S instead of S makes every sign fall on an FMA operand.  After the 2*NT steps the tiles hold inv(S) and v holds
// inv(S)*v (v rides through the sweeps as a fifth column, so no mat-vec is needed).  Operand traffic per lane: 8 fragment
// doubles per FOUR pivots (the rank-1 register sweep above needs 32 per ONE pivot, which made it shared-memory bound);
// symmetry halves the FP64 work.
// Shared scratch per warp: Ps, Ws = 4 column planes of PLANE doubles each ([col][row]: conflict-free for the row-wise,
// fragment-wise and tile-wise accesses), vs = 32 doubles.  `ok` is uniform across the warp.
__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// 1/x for a positive, finite, normal x: hardware seed (~2^-20) + one cubic Newton step, three dependent FMAs
// (relative error ~2^-60; no special-case slow path, the callers have already rejected non-positive / non-finite pivots)
__device__ __forceinline__ double rcp_pos(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x, y, 1.0);
    const double t = fma(e, e, e);
    return fma(y, t, y);
}
// positive, finite and not denormal / huge, tested on the exponent word (integer pipe, keeps the FP64 pipe for the math)
__device__ __forceinline__ bool pivot_ok(double x) {
    return (unsigned)(__double2hiint(x) - 0x00100000) < (unsigned)(0x7e300000 - 0x00100000);
}
// -x through the integer pipe (sign-bit flip): keeps negations that must be materialised off the FP64 pipe
__device__ __forceinline__ double neg_alu(double x) { return __hiloint2double(__double2hiint(x) ^ 0x80000000, __double2loint(x)); }
__host__ __device__ constexpr int tri_idx(int ti, int tj, int NT) { return ti * NT - ti * (ti - 1) / 2 + (tj - ti); }
constexpr int GJ_PLANE = 36;                    // plane stride of the panel buffers: 32 rows + 4 (bank skew between the 4 columns)
constexpr int GJ_SCRATCH = 8 * GJ_PLANE + 32;   // doubles of scratch per warp: Ps | Ws | vs

// One block step's lane = row work, shared by the warp-level and the CTA-level inverse: the four sweeps on this lane's panel
// row y[0..3] (and rhs v), driven by the 4 x 4 pivot block a[][] / rhs pivots vk[] that the lane evolves itself.
// In: y = row of the panel of T = -S, a = rows 4s..4s+3 of the panel, `prow` = this lane's row index - 4s (0..3 on a pivot row).
// Out: gq = multipliers (A fragment values), pq = column entries before their sweep (+1 on the pivot entry; B fragment values).
__device__ __forceinline__ bool gj_panel_sweeps(double (&a)[4][4], double (&vk)[4], double (&y)[4], double& v, const int prow,
                                                double (&gq)[4], double (&pq)[4]) {
    bool ok = true;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        const double dpiv = neg_alu(a[cc][cc]);                 // the pivot of S
        ok = ok && pivot_ok(dpiv);
        const double id = rcp_pos(dpiv);
        const bool piv = prow == cc;
        // x[q] -= f*x_piv[q] with f = x[cc]/d (f = 1 - 1/d on the pivot row itself, whose entries equal the pivot row's);
        // in terms of y = -x:  y[q] += g*pr[q], g = -f = y[cc]/d (pivot row: 1/d - 1);  v -= f*v_piv = v + g*v_piv
        const double g = piv ? id - 1.0 : y[cc] * id;
        pq[cc] = piv ? y[cc] + 1.0 : y[cc];
        gq[cc] = g;
#pragma unroll
        for (int q = 0; q < 4; ++q) if (q != cc) y[q] = fma(g, a[cc][q], y[q]);
        v = fma(g, vk[cc], v);
        y[cc] = piv ? id : g;
        // the later pivot rows (and rhs pivots) of the block
#pragma unroll
        for (int i = cc + 1; i < 4; ++i) {
            const double gi = a[i][cc] * id;
#pragma unroll
            for (int q = 0; q < 4; ++q) if (q != cc) a[i][q] = fma(gi, a[cc][q], a[i][q]);
            vk[i] = fma(gi, vk[cc], vk[i]);
            a[i][cc] = gi;
        }
    }
    return ok;
}

template <int NT>
__device__ __forceinline__ bool warp_block_gj_sym(double (&c)[NT * (NT + 1) / 2][2], double& v, const int lane,
                                                  double* __restrict__ scr) {
    constexpr int N = 8 * NT, PL = GJ_PLANE;
    double* Ps = scr;
    double* Ws = scr + 4 * PL;
    double* vs = scr + 8 * PL;
    const int r = lane >> 2, j = lane & 3;
    const bool rowlane = lane < N;
    bool ok = true;
#pragma unroll
    for (int s = 0; s < 2 * NT; ++s) {
        const int tk = s >> 1, half = s & 1;
        // 1. publish the column panel of T = -S (plane [col][row]) and the rhs
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            if (t <= tk) {
                if ((j >> 1) == half) {
                    Ps[(2 * (j & 1)) * PL + 8 * t + r] = c[tri_idx(t, tk, NT)][0];
                    Ps[(2 * (j & 1) + 1) * PL + 8 * t + r] = c[tri_idx(t, tk, NT)][1];
                }
            } else {
                if ((r >> 2) == half) {
                    Ps[(r & 3) * PL + 8 * t + 2 * j] = c[tri_idx(tk, t, NT)][0];
                    Ps[(r & 3) * PL + 8 * t + 2 * j + 1] = c[tri_idx(tk, t, NT)][1];
                }
            }
        }
        vs[lane] = v;
        __syncwarp();
        // 2. lane = row
        double a[4][4], vk[4], y[4] = {0.0, 0.0, 0.0, 0.0}, gq[4], pq[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double2 lo = *reinterpret_cast<const double2*>(Ps + q * PL + 4 * s), hi = *reinterpret_cast<const double2*>(Ps + q * PL + 4 * s + 2);
            a[0][q] = lo.x; a[1][q] = lo.y; a[2][q] = hi.x; a[3][q] = hi.y;
        }
        {
            const double2 lo = *reinterpret_cast<const double2*>(vs + 4 * s), hi = *reinterpret_cast<const double2*>(vs + 4 * s + 2);
            vk[0] = lo.x; vk[1] = lo.y; vk[2] = hi.x; vk[3] = hi.y;
        }
        if (rowlane) {
#pragma unroll
            for (int q = 0; q < 4; ++q) y[q] = Ps[q * PL + lane];
        }
        ok = gj_panel_sweeps(a, vk, y, v, lane - 4 * s, gq, pq) && ok;
        __syncwarp();                                   // every lane has read the pivot block before rows are overwritten
        if (rowlane) {
#pragma unroll
            for (int q = 0; q < 4; ++q) { Ws[q * PL + lane] = gq[q]; Ps[q * PL + lane] = pq[q]; }
        }
        __syncwarp();
        // 3. fragments and the rank-4 update of every stored tile
        double pf[NT], wf[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) { pf[t] = Ps[j * PL + 8 * t + r]; wf[t] = Ws[j * PL + 8 * t + r]; }
#pragma unroll
        for (int ti = 0; ti < NT; ++ti)
#pragma unroll
            for (int tj = ti; tj < NT; ++tj) dmma884(c[tri_idx(ti, tj, NT)], wf[ti], pf[tj]);
        if ((r >> 2) == half && j == (r >> 1)) {
            if (r & 1) c[tri_idx(tk, tk, NT)][1] += 2.0; else c[tri_idx(tk, tk, NT)][0] += 2.0;
        }
        __syncwarp();
    }
    return ok;
}

// CTA version: thread t owns elements e = t + q*blockDim.x (q < Q) of the row-major H x H matrix; column k travels
// through a double-buffered shared vector, one __syncthreads per sweep.  cbuf = 2*H doubles, sbuf = H doubles.
// Result stays in a[]; `ok` is uniform across the CTA.
template <int Q>
__device__ __forceinline__ bool block_spd_inverse_reg(double (&a)[Q], const int (&eij)[Q], int H, double* cbuf, double* sbuf) {
    // eij[q] = row | (col << 8) of the owned element, -1 when the slot is unused (H <= 128)
    bool ok = true;
#pragma unroll
    for (int q = 0; q < Q; ++q) if (eij[q] >= 0 && (eij[q] & 255) == (eij[q] >> 8)) sbuf[eij[q] & 255] = 1.0 / sqrt(a[q]);
    __syncthreads();
#pragma unroll
    for (int q = 0; q < Q; ++q) if (eij[q] >= 0) a[q] *= sbuf[eij[q] & 255] * sbuf[eij[q] >> 8];
    for (int k = 0; k < H; ++k) {
        double* col = cbuf + (k & 1) * H;
#pragma unroll
        for (int q = 0; q < Q; ++q) if ((eij[q] >> 8) == k) col[eij[q] & 255] = a[q];
        __syncthreads();
        const double d = col[k];
        if (!(d > 0.0) || !(d < 1e300)) ok = false;
        const double id = 1.0 / d;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            if (eij[q] >= 0) {
                const int i = eij[q] & 255, j = eij[q] >> 8;
                double v;
                if (i == k) v = (j == k) ? -id : col[j] * id;
                else if (j == k) v = col[i] * id;
                else v = a[q] - (col[i] * col[j]) * id;
                a[q] = v;
            }
        }
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) if (eij[q] >= 0) a[q] = -a[q] * sbuf[eij[q] & 255] * sbuf[eij[q] >> 8];
    return ok;
}

// Largest eigenvalue of the symmetric matrix A (n x n, full storage, row stride ld, shared memory; destroyed) by
// Householder tridiagonalisation followed by parallel multisection on the Sturm sequence: orthogonal similarity +
// bisection, so lambda_max carries an absolute error of a few ulp of ||A|| (what LAPACK's SVD gives the reference for
// norm(::Matrix)).  work = 4*n doubles.  Whole CTA (blockDim.x >= 64, multiple of 32); result valid in every thread.
// A is first scaled by 2^-e so that its largest entry lies in [1/2, 1), and lambda is scaled back by 2^e: the Sturm
// recurrence is division-free and would overflow or underflow for entries beyond about 1e+-77.  The scale itself is exact and
// every input scale then runs on the same matrix, but the every-4-steps rescale picks max(|p_{i-1}|, |p_i|), whose winner
// depends on the scale, so against the unscaled recurrence lambda may move in its last bits.  An all-zero matrix gives
// exactly 0.
__device__ inline double sym_lambda_max(double* A, int ld, int n, double* work) {
    const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, warp = t >> 5;
    double* dv = work;            // diagonal of T
    double* ev = work + n;        // sub-diagonal of T (ev[k] couples k and k+1)
    double* v = work + 2 * n;     // Householder vector
    double* p = work + 3 * n;     // p / q vector
    __shared__ double s_sc[4];    // beta, alpha, K, flag
    __shared__ double s_lo, s_hi;
    __shared__ int s_first;
    __shared__ unsigned long long s_amax;   // bit pattern of max |A_ij| (non-negative doubles order as their bit patterns)
    if (n <= 0) return 0.0;
    if (t == 0) s_amax = 0ull;
    // NaN / Inf anywhere -> NaN (the reference's norm would propagate it)
    int bad = 0;
    double amax = 0.0;
    for (int e = t; e < n * n; e += nt) {
        const double x = A[(e / n) * ld + (e % n)];
        if (!(fabs(x) <= 1.79e308)) bad = 1;
        else amax = fmax(amax, fabs(x));
    }
    if (__syncthreads_or(bad)) return nan("");
    if (n == 1) return A[0];
    atomicMax(&s_amax, (unsigned long long)__double_as_longlong(amax));
    __syncthreads();
    const double big = __longlong_as_double((long long)s_amax);
    if (big == 0.0) return 0.0;
    int escale;
    frexp(big, &escale);
    for (int e = t; e < n * n; e += nt) { double* x = A + (e / n) * ld + (e % n); *x = ldexp(*x, -escale); }
    __syncthreads();
    for (int k = 0; k < n - 2; ++k) {
        const int m = n - k - 1;                  // trailing block is rows/cols k+1 .. n-1
        double* Asub = A + (k + 1) * ld + (k + 1);
        if (warp == 0) {                          // x = A[k+1:, k] ; v = x - alpha*e1 ; beta = 2/(v'v)
            double s = 0.0;
            for (int i = lane; i < m; i += 32) { const double x = A[(k + 1 + i) * ld + k]; v[i] = x; s = fma(x, x, s); }
            s = warp_sum(s);
            __syncwarp();
            const double x0 = v[0];
            const double tail = s - x0 * x0;      // sum of squares below the first entry
            if (lane == 0) {
                if (!(tail > 0.0)) { s_sc[0] = 0.0; s_sc[1] = x0; }          // already tridiagonal in this column
                else {
                    const double alpha = (x0 >= 0.0) ? -sqrt(s) : sqrt(s);
                    const double v0 = x0 - alpha;
                    v[0] = v0;
                    s_sc[0] = 2.0 / (tail + v0 * v0);
                    s_sc[1] = alpha;
                }
            }
        }
        __syncthreads();
        const double beta = s_sc[0];
        if (beta != 0.0) {
            // p = beta * Asub * v : TPR threads per row, partial dots combined by shuffles (column access: A is symmetric)
            {
                const int TPR = 8, row = t / TPR, sub = t % TPR;
                for (int r0 = 0; r0 < m; r0 += nt / TPR) {
                    const int i = r0 + row;
                    double s = 0.0;
                    if (i < m) for (int j = sub; j < m; j += TPR) s = fma(Asub[j * ld + i], v[j], s);
                    s += __shfl_xor_sync(0xffffffffu, s, 1);
                    s += __shfl_xor_sync(0xffffffffu, s, 2);
                    s += __shfl_xor_sync(0xffffffffu, s, 4);
                    if (i < m && sub == 0) p[i] = beta * s;
                }
            }
            __syncthreads();
            if (warp == 0) {                      // K = beta/2 * p'v ; q = p - K v
                double s = 0.0;
                for (int i = lane; i < m; i += 32) s = fma(p[i], v[i], s);
                s = warp_sum(s);
                const double K = 0.5 * beta * s;
                for (int i = lane; i < m; i += 32) p[i] -= K * v[i];
            }
            __syncthreads();
            // Asub -= v q' + q v'  (2-D thread mapping, no integer division)
            for (int i = warp; i < m; i += nt / 32) {
                const double vi = v[i], pi = p[i];
                for (int j = lane; j < m; j += 32) Asub[i * ld + j] -= vi * p[j] + pi * v[j];
            }
        }
        if (t == 0) { dv[k] = A[k * ld + k]; ev[k] = s_sc[1]; }
        __syncthreads();
    }
    if (t == 0) {
        dv[n - 2] = A[(n - 2) * ld + (n - 2)];
        dv[n - 1] = A[(n - 1) * ld + (n - 1)];
        ev[n - 2] = A[(n - 1) * ld + (n - 2)];
        double lo = 1e308, hi = -1e308;           // Gershgorin interval
        for (int i = 0; i < n; ++i) {
            const double r = (i > 0 ? fabs(ev[i - 1]) : 0.0) + (i < n - 1 ? fabs(ev[i]) : 0.0);
            lo = fmin(lo, dv[i] - r); hi = fmax(hi, dv[i] + r);
        }
        const double pad = 4e-16 * fmax(fabs(lo), fabs(hi)) + 1e-300;
        s_lo = lo - pad; s_hi = hi + pad;
    }
    __syncthreads();
    // multisection: count(x) = #eigenvalues < x = sign changes of the Sturm sequence p_0 = 1, p_1 = d_0 - x,
    // p_{i+1} = (d_i - x) p_i - e_{i-1}^2 p_{i-1} (division-free; rescaled every 4 steps); lambda_max is where count
    // steps from n-1 to n.  Every thread evaluates one sample point per round, the bracket shrinks (blockDim+1)-fold.
    double* ev2 = v;                              // v, p are free after the tridiagonalisation
    for (int i = t; i < n - 1; i += nt) ev2[i] = ev[i] * ev[i];
    __syncthreads();
    for (int iter = 0; iter < 12; ++iter) {
        const double lo = s_lo, hi = s_hi;
        if (!(hi - lo > 2e-15 * fmax(fabs(lo), fabs(hi)))) break;
        const double x = lo + (hi - lo) * ((double)(t + 1) / (double)(nt + 1));
        double pm = 1.0, pc = dv[0] - x;
        int cnt = pc < 0.0;
        for (int i = 1; i < n; ++i) {
            const double pn = (dv[i] - x) * pc - ev2[i - 1] * pm;
            // sign change between pc and pn (a zero inherits the previous sign)
            const double sc_ = (pc != 0.0) ? pc : pm;
            cnt += ((pn < 0.0) != (sc_ < 0.0)) && (pn != 0.0);
            pm = (pc != 0.0) ? pc : pm * 1e-300;          // keep the sign information of pm when pc vanished
            pc = pn;
            if ((i & 3) == 0) {                           // rescale: only ratios and signs matter
                const double sc = fmax(fabs(pm), fabs(pc));
                if (sc > 0.0 && sc < 1e308) { const double r = 1.0 / sc; pm *= r; pc *= r; }
            }
        }
        if (t == 0) s_first = nt;
        __syncthreads();
        if (cnt == n) atomicMin(&s_first, t);     // smallest sample point that lies above every eigenvalue
        __syncthreads();
        const int f = s_first;
        __syncthreads();
        if (t == 0) {
            const double w = (hi - lo) / (double)(nt + 1);
            s_hi = (f < nt) ? lo + w * (double)(f + 1) : hi;
            s_lo = (f > 0) ? lo + w * (double)f : lo;
        }
        __syncthreads();
    }
    return ldexp(0.5 * (s_lo + s_hi), escale);
}

}  // namespace vb
