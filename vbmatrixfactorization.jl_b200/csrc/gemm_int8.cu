// K1 / K2 on the INT8 tensor cores (tcgen05.mma.kind::i8) with exact slice splitting, for H <= 64.
//
// Both operands are written as seven signed radix-256 digits with power-of-two scales (the Ozaki scheme):
//   Y = diag(2^F) * Z * diag(2^E),  Z = sum_{i<7} 2^-(7+8i) S_i + r,  -128 <= S_i <= 127, |r| <= 2^-56
// F_l is the exponent of the row maximum of Y.  E_m is the smallest exponent with |row-scaled Y| <= (127/128) 2^E_m over the
// column, so |Z| <= 127/128 and rint(Z * 2^55) lies inside the range of seven balanced digits, whose positive end is only
// 127 (2^56 - 1) / 255.  The small operand of a contraction (BHat for K1, AHat for K2) is scaled by the same exponents
// (diag(2^F) * B, diag(2^E) * A), given one exponent per column (K2: per column and split-K chunk) under the same 127/128
// rule and cut the same way.  Every digit is a plain int8, so signed kind::i8 multiplies them as they are.  The digit
// products S_i * T_j with i + j = k form level k; levels 0..6 (28 products) are accumulated exactly in INT32 tensor memory and
// combined in FP64:
//   sum_k 2^-(8k+14) * level_k,  levels 6 down to 0,  times 2^(row exponent + column exponent).
// Y's digits are built once per attached Y (i8_build_Y); the small operand is cut every iteration (i8_slice_B / _A).
//
// Tensor memory: level k of the 128 x Hp tile lives in columns [Hp*k, Hp*(k+1)) (Hp = H rounded up to 16, <= 64, at most 448
// of the 512 columns allocated).  For Y digit i, ONE run of MMAs takes the operand digits j = 0..6-i, laid side by side along
// N in shared memory, and writes columns [Hp*i, Hp*7): every level the digit contributes to in one instruction stream (N
// split in pieces <= 256: 10 MMAs per stage at Hp = 64).  Level 6 sums 7 products of |S| <= 128 per k (114688), so INT32
// holds 18724 k; the accumulators are flushed every 16384 k.
//
// Pipeline (one CTA per SM): warp 4 issues TMA loads of 32 k of all 7 Y digit planes and all 7 operand planes per stage into
// a STAGES-deep ring guarded by full / empty mbarriers, one lane of warp 5 issues the MMAs and commits each stage back, warps
// 0-3 read tensor memory (warp q owns lanes 32q..32q+31 = tile rows) and write the FP64 result.  Persistent CTAs walk a
// static list of (tile, split) work items; split-K slabs are summed in fixed order by the caller, so results are
// bit-reproducible.
//   K1  P = Y' * B:  A operand = Y digits, K-major (rows m, k = l), box {32, 128, 7}, 32-byte swizzle.
//   K2  Q = Y  * A:  A operand = the same digits read MN-major (rows l, k = m), box {128, 32, 7}, 128-byte swizzle.
//   The B operand is the small operand's digits, K-major [7][Hp][ld], box {32, Hp, 7}, 32-byte swizzle.
#include "gemm.cuh"
#include <algorithm>

namespace vb {
namespace i8k {

constexpr int TM = 128;                 // tile rows (MMA M)
constexpr int KB = 32;                  // k per stage = K of one int8 MMA
constexpr int NSL = I8_NSL;             // digit planes per operand
constexpr int STAGES = 4;               // measured a little faster than 5 stages (which also fit) at config 3
constexpr int A_BYTES = NSL * TM * KB;  // 28 KB: 7 digits x 128 rows x 32 k
constexpr int B_BYTES = NSL * 64 * KB;  // 14 KB at Hp = 64
constexpr int SB = A_BYTES + B_BYTES;   // 42 KB: stage and plane offsets stay 1024-aligned for the 128-byte swizzle
static_assert(SB % 1024 == 0 && A_BYTES % 1024 == 0, "stage layout must stay 1024-byte aligned");
constexpr int SMEM = STAGES * SB + 1024 + 256;
static_assert(SMEM <= 227 * 1024, "stage ring exceeds the shared memory of one CTA");
constexpr int SEG_KB = 16384 / KB;      // k-blocks per flush: level 6 stays below 2^31
static_assert((long long)SEG_KB * KB * NSL * 128 * 128 < (1ll << 31), "level 6 may overflow INT32 between flushes");
constexpr int EXP_NONE = -(1 << 30);    // exponent of 0 (and of non-finite values): below every real exponent
constexpr int EXP_NAN = 1 << 30;        // operand column exponent of a column with a non-finite value: above every real one

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_i8(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor (sm_100): start, leading / stride byte offsets (16-byte units), version 1, layout type
__device__ __forceinline__ uint64_t sdesc(uint32_t addr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46) |
           ((uint64_t)layout << 61);
}
constexpr uint32_t LAYOUT_SW128 = 2, LAYOUT_SW32 = 6;

__device__ __forceinline__ int exp_of(double x) {
    if (x == 0.0 || !isfinite(x)) return EXP_NONE;
    int e;
    frexp(x, &e);
    return e;
}
// smallest e with |x| <= (127/128) 2^e: frexp's exponent, plus one when the mantissa exceeds 127/128 (monotonic in |x|)
__device__ __forceinline__ int exp_digits(double x) {
    if (x == 0.0 || !isfinite(x)) return EXP_NONE;
    int e;
    const double m = frexp(x, &e);
    return fabs(m) > 127.0 / 128.0 ? e + 1 : e;
}
__device__ __forceinline__ int exp_fix(int e) { return e <= EXP_NONE ? 0 : e; }

// rint(x * 2^(55 - e)): the digits' fixed-point form of w = x * 2^-e (|w| <= 127/128, so |result| <= 127 * 2^48).
// Non-finite values get zero digits; the outputs they reach are set to NaN from the flags instead.
__device__ __forceinline__ long long fixed55(double x, int e) { return isfinite(x) ? __double2ll_rn(ldexp(x, 55 - e)) : 0ll; }

// seven balanced radix-256 digits of X = rint(w * 2^55): w = sum_i d_i 2^-(7+8i), d_i in [-128, 127], taken from the bottom.
// The digit is the low byte read as signed; X - d is then a multiple of 256.  Four consecutive values per 32-bit word: byte q
// of word i = digit i of x[q].
__device__ __forceinline__ void digits4(const long long (&x)[4], uint32_t (&out)[NSL]) {
#pragma unroll
    for (int i = 0; i < NSL; ++i) out[i] = 0u;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        long long t = x[q];
#pragma unroll
        for (int i = NSL - 1; i >= 0; --i) {
            const int d = (int8_t)(t & 255);
            out[i] |= ((uint32_t)t & 0xffu) << (8 * q);
            t = (t - d) >> 8;
        }
    }
}

__device__ __forceinline__ int block_max_int(int v, int* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    if (w == 0) {
        v = l < (int)(blockDim.x >> 5) ? red[l] : EXP_NONE;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
        if (l == 0) red[0] = v;
    }
    __syncthreads();
    return red[0];
}

// ------------------------------------------------------------------------------------------- slices of Y (once per attach)
// F_l = frexp exponent of the row maximum over the finite values; Fbad[l] = 1 when row l holds a NaN or Inf (zeroed before)
__global__ void __launch_bounds__(256) y_row_exp_kernel(const double* __restrict__ Y, int ldY, int L, int M, int* __restrict__ F,
                                                        int* __restrict__ Fbad) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    int e = EXP_NONE;
    bool bad = false;
    for (int m = blockIdx.y; m < M; m += gridDim.y) {
        const double y = Y[(size_t)m * ldY + l];
        e = max(e, exp_of(y));
        bad |= !isfinite(y);
    }
    atomicMax(F + l, e);
    if (bad) Fbad[l] = 1;
}

// one CTA per column m: E_m over the finite values and Ebad[m] (column m holds a NaN or Inf), then the column's seven digit
// planes (4 rows per thread and 32-bit word)
__global__ void __launch_bounds__(256) y_slices_kernel(const double* __restrict__ Y, int ldY, int L, int M, const int* __restrict__ F,
                                                       int* __restrict__ E, int* __restrict__ Ebad, uint8_t* __restrict__ Z, int ldZ) {
    __shared__ int red[32];
    const int m = blockIdx.x;
    const double* y = Y + (size_t)m * ldY;
    int e = EXP_NONE, bad = 0;
    for (int l = threadIdx.x; l < L; l += blockDim.x) {
        const int ey = exp_digits(y[l]);
        if (ey > EXP_NONE) e = max(e, ey - exp_fix(F[l]));
        bad |= !isfinite(y[l]);
    }
    bad = __syncthreads_or(bad);
    const int Em = exp_fix(block_max_int(e, red));
    if (threadIdx.x == 0) { E[m] = Em; Ebad[m] = bad; }
    const size_t plane = (size_t)M * ldZ;
    for (int l4 = threadIdx.x; l4 < ldZ / 4; l4 += blockDim.x) {
        long long x[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int l = 4 * l4 + q;
            x[q] = l < L ? fixed55(y[l], exp_fix(F[l]) + Em) : 0;
        }
        uint32_t s[NSL];
        digits4(x, s);
#pragma unroll
        for (int i = 0; i < NSL; ++i) reinterpret_cast<uint32_t*>(Z + i * plane + (size_t)m * ldZ)[l4] = s[i];
    }
}

// ------------------------------------------------------------------------------------------- K1 operand: digits of diag(2^F) B
// one CTA per column h < Hp (rows h >= H are zero): G_h (EXP_NAN when the column holds a NaN or Inf), then the column's
// digits, layout [7][Hp][ldZ]
__global__ void __launch_bounds__(512) b_slices_kernel(const double* __restrict__ B, int ldB, int L, int H, int Hp, const int* __restrict__ F,
                                                       uint8_t* __restrict__ W, int ldZ, int* __restrict__ G, const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    __shared__ int red[32];
    const int h = blockIdx.x;
    const double* b = B + (size_t)h * ldB;
    int e = EXP_NONE, bad = 0;
    if (h < H)
        for (int l = threadIdx.x; l < L; l += blockDim.x) {
            const int eb = exp_digits(b[l]);
            if (eb > EXP_NONE) e = max(e, eb + exp_fix(F[l]));
            bad |= !isfinite(b[l]);
        }
    bad = __syncthreads_or(bad);
    const int Gh = bad ? EXP_NAN : exp_fix(block_max_int(e, red));
    if (threadIdx.x == 0) G[h] = Gh;
    const size_t plane = (size_t)Hp * ldZ;
    for (int l4 = threadIdx.x; l4 < ldZ / 4; l4 += blockDim.x) {
        long long x[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int l = 4 * l4 + q;
            x[q] = (h < H && l < L) ? fixed55(b[l], Gh - exp_fix(F[l])) : 0;
        }
        uint32_t s[NSL];
        digits4(x, s);
#pragma unroll
        for (int i = 0; i < NSL; ++i) reinterpret_cast<uint32_t*>(W + i * plane + (size_t)h * ldZ)[l4] = s[i];
    }
}

// ------------------------------------------------------------------------------------------- K2 operand: digits of diag(2^E) A
// A is [M][H] (row m contiguous in h).  Exponents per (split-K chunk, column): G[c][h] = max over m in chunk c (atomicMax on
// integers: order-independent), EXP_NAN when the chunk of the column holds a NaN or Inf.  256 rows per CTA, thread =
// (h = t % 64, rows t / 64 + 4 r).
__global__ void __launch_bounds__(256) a_exp_kernel(const double* __restrict__ A, int M, int H, int Hp, const int* __restrict__ E, int kchunk,
                                                    int* __restrict__ G, const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    const int h = threadIdx.x & 63;
    if (h >= H) return;
    const int m0 = blockIdx.x * 256, m1 = min(M, m0 + 256);
    int cur = -1, e = EXP_NONE;
    for (int m = m0 + (threadIdx.x >> 6); m < m1; m += 4) {
        const int c = m / kchunk;
        if (c != cur) {
            if (cur >= 0 && e > EXP_NONE) atomicMax(G + cur * Hp + h, e);
            cur = c; e = EXP_NONE;
        }
        const double a = A[(size_t)m * H + h];
        const int ea = exp_digits(a);
        if (!isfinite(a)) e = EXP_NAN;
        else if (ea > EXP_NONE) e = max(e, ea + E[m]);
    }
    if (cur >= 0 && e > EXP_NONE) atomicMax(G + cur * Hp + h, e);
}

// 64 rows per CTA through shared memory; output K-major [7][Hp][ldM]
__global__ void __launch_bounds__(256) a_slices_kernel(const double* __restrict__ A, int M, int H, int Hp, const int* __restrict__ E, int kchunk,
                                                       const int* __restrict__ G, uint8_t* __restrict__ W, int ldM, const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    __shared__ double tile[64 * 64];
    const int m0 = blockIdx.x * 64;
    const int nm = min(64, M - m0);
    for (int t = threadIdx.x; t < nm * H; t += blockDim.x) tile[t] = A[(size_t)m0 * H + t];
    __syncthreads();
    const size_t plane = (size_t)Hp * ldM;
    for (int t = threadIdx.x; t < Hp * 16; t += blockDim.x) {
        const int h = t >> 4, g = t & 15;
        if (m0 + 4 * g >= ldM) continue;
        long long x[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = 4 * g + q, m = m0 + r;
            x[q] = 0;
            if (h < H && r < nm) x[q] = fixed55(tile[r * H + h], exp_fix(G[(m / kchunk) * Hp + h]) - E[m]);
        }
        uint32_t s[NSL];
        digits4(x, s);
#pragma unroll
        for (int i = 0; i < NSL; ++i) reinterpret_cast<uint32_t*>(W + i * plane + (size_t)h * ldM + m0)[g] = s[i];
    }
}

// ------------------------------------------------------------------------------------------- the contraction
// Work item w: tile = w % ntile (128 output rows), split s = w / ntile (k range [s*klen, min(kdim, (s+1)*klen)), klen a
// multiple of 32).  Output element (row, h) of slab s: out[s*slab + row*rs + h*hs] = 2^(rowexp[row] + colexp[s*cstride + h])
// * sum over the k range, or NaN when rowbad[row] is set or the column exponent is EXP_NAN (a non-finite input reaches the
// element); rows >= nrows and h >= H are not written.
template <bool MN>
__global__ void __launch_bounds__(192, 1)
gemm_i8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, double* __restrict__ out,
               int nrows, int kdim, int S, int klen, int H, int Hp, const int* __restrict__ rowexp,
               const int* __restrict__ rowbad, const int* __restrict__ colexp, int cstride, size_t slab, size_t rs, size_t hs, const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t full0 = base + STAGES * SB, empty0 = full0 + STAGES * 8;
    const uint32_t tfull = empty0 + STAGES * 8, tempty = tfull + 8, tslot = tempty + 8;
    uint32_t* tslot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tslot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t ncols = Hp * NSL <= 128 ? 128 : (Hp * NSL <= 256 ? 256 : 512);
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tslot_ptr);

    const int ntile = (nrows + TM - 1) / TM;
    const int nwork = ntile * S;
    const uint32_t tx_bytes = A_BYTES + NSL * Hp * KB;

    if (warp == 4) {  // ---------------- TMA producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int r0 = (w % ntile) * TM, k0 = (w / ntile) * klen, k1 = min(kdim, k0 + klen);
                for (int k = k0; k < k1; k += KB, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    mbar_expect_tx(full0 + 8 * s, tx_bytes);
                    if (MN) tma_load_3d(base + s * SB, &tmA, full0 + 8 * s, r0, k, 0);
                    else tma_load_3d(base + s * SB, &tmA, full0 + 8 * s, k, r0, 0);
                    tma_load_3d(base + s * SB + A_BYTES, &tmB, full0 + 8 * s, k, 0, 0);
                }
            }
        }
    } else if (warp == 5) {  // ---------------- MMA issuer
        if (lane == 0) {
            // instruction descriptor: S32 accumulator, signed A and B, A major (K2: MN), B K-major, M = 128
            const uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((MN ? 1u : 0u) << 15) | ((uint32_t)(TM >> 4) << 24);
            uint32_t it = 0, sg = 0;
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int k0 = (w / ntile) * klen, k1 = min(kdim, k0 + klen);
                const int nkb = (k1 - k0 + KB - 1) / KB;
                for (int kb0 = 0; kb0 < nkb; kb0 += SEG_KB, ++sg) {
                    const int kb1 = min(nkb, kb0 + SEG_KB);
                    mbar_wait(tempty, (sg & 1) ^ 1);
                    tc_fence_after();
                    for (int kb = kb0; kb < kb1; ++kb, ++it) {
                        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
                        mbar_wait(full0 + 8 * s, ph);
                        tc_fence_after();
                        const uint32_t a0 = base + s * SB, b0 = a0 + A_BYTES;
#pragma unroll
                        for (int i = 0; i < NSL; ++i) {
                            const uint64_t ad = MN ? sdesc(a0 + i * (TM * KB), 16, 1024, LAYOUT_SW128)
                                                   : sdesc(a0 + i * (TM * KB), 16, 256, LAYOUT_SW32);
                            const int ntot = Hp * (NSL - i);
                            for (int p = 0; p < ntot; p += 256) {
                                const int n = min(256, ntot - p);
                                const uint64_t bd = sdesc(b0 + p * KB, 16, 256, LAYOUT_SW32);
                                mma_i8(tmem + Hp * i + p, ad, bd, idesc0 | ((uint32_t)(n >> 3) << 17), (kb > kb0 || i > 0) ? 1u : 0u);
                            }
                        }
                        tc_commit(empty0 + 8 * s);
                    }
                    tc_commit(tfull);
                }
            }
        }
    } else {  // ---------------- epilogue: warp q reads tensor-memory lanes 32q..32q+31
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        uint32_t sg = 0;
        for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
            const int tile = w % ntile, sp = w / ntile;
            const int k0 = sp * klen, k1 = min(kdim, k0 + klen);
            const int nkb = (k1 - k0 + KB - 1) / KB;
            const int row = tile * TM + warp * 32 + lane;
            const bool live = row < nrows;
            const int re = live ? rowexp[row] : 0;
            const bool bad = live && rowbad[row] != 0;
            double* o = out + (size_t)sp * slab + (size_t)(live ? row : 0) * rs;
            const int* ce = colexp + (size_t)sp * cstride;
            for (int kb0 = 0; kb0 < nkb; kb0 += SEG_KB, ++sg) {
                mbar_wait(tfull, sg & 1);
                tc_fence_after();
                for (int h0 = 0; h0 < Hp; h0 += 8) {
                    uint32_t v[NSL][8];
#pragma unroll
                    for (int k = 0; k < NSL; ++k) tmem_ld8(tmem + lane_base + Hp * k + h0, v[k]);
                    tmem_wait_ld();
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int h = h0 + c;
                        // levels 6 down to 0: acc = sum_k level_k * 2^-8k (every step exact up to one rounding)
                        double acc = (double)(int)v[NSL - 1][c];
#pragma unroll
                        for (int k = NSL - 2; k >= 0; --k) acc = fma(acc, 0x1p-8, (double)(int)v[k][c]);
                        if (live && h < H) {
                            const double x = (bad || ce[h] == EXP_NAN) ? __longlong_as_double(0x7ff8000000000000ll)
                                                                       : ldexp(acc, re + ce[h] - 14);
                            double* p = o + (size_t)h * hs;
                            *p = kb0 == 0 ? x : *p + x;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(ncols) : "memory");
    }
}

}  // namespace i8k
using namespace i8k;

// ------------------------------------------------------------------------------------------- host side
int make_tmap_3d_i8(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2,
                    uint32_t b0, uint32_t b1, uint32_t b2, bool swizzle128) {
    PFN_encodeTiled enc = tmap_encoder();
    if (!enc) return -1;
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (s1 & 15) != 0 || (s2 & 15) != 0) {
        set_error("INT8 tensor map needs a 16-byte aligned base and pitches (base=%p pitches %llu, %llu)", base,
                  (unsigned long long)s1, (unsigned long long)s2);
        return -1;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {s1, s2};
    cuuint32_t box[3] = {b0, b1, b2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (int8) failed with CUresult %d (dims %llu x %llu x %llu, box %u x %u x %u)", (int)r,
                  (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, b0, b1, b2);
        return -1;
    }
    return 0;
}

int gemm_i8_init_device() {
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_i8_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_i8_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    return 0;
}

int i8_build_Y(cudaStream_t st, const double* Y, int ldY, int L, int M, uint8_t* Z, int ldZ, int* F, int* E, int* Fbad, int* Ebad) {
    if (L <= 0 || M <= 0) return 0;
    VB_CUDA_OK(cudaMemsetAsync(F, 0x80, (size_t)L * 4, st));
    VB_CUDA_OK(cudaMemsetAsync(Fbad, 0, (size_t)L * 4, st));
    dim3 g1((L + 255) / 256, std::min(M, 512));
    y_row_exp_kernel<<<g1, 256, 0, st>>>(Y, ldY, L, M, F, Fbad);
    VB_LAUNCH_OK();
    y_slices_kernel<<<M, 256, 0, st>>>(Y, ldY, L, M, F, E, Ebad, Z, ldZ);
    VB_LAUNCH_OK();
    return 0;
}

int i8_slice_B(cudaStream_t st, const double* B, int ldB, int L, int H, const int* F, uint8_t* W, int ldZ, int* G, const Scalars* sc) {
    const int Hp = i8_hpad(H);
    b_slices_kernel<<<Hp, 512, 0, st>>>(B, ldB, L, H, Hp, F, W, ldZ, G, sc);
    VB_LAUNCH_OK();
    return 0;
}

int i8_slice_A(cudaStream_t st, const double* A, int M, int H, const int* E, int kchunk, int S, uint8_t* W, int ldM, int* G, const Scalars* sc) {
    if (M <= 0) return 0;
    const int Hp = i8_hpad(H);
    VB_CUDA_OK(cudaMemsetAsync(G, 0x80, (size_t)S * Hp * 4, st));
    a_exp_kernel<<<(M + 255) / 256, 256, 0, st>>>(A, M, H, Hp, E, kchunk, G, sc);
    VB_LAUNCH_OK();
    a_slices_kernel<<<(ldM + 63) / 64, 256, 0, st>>>(A, M, H, Hp, E, kchunk, G, W, ldM, sc);
    VB_LAUNCH_OK();
    return 0;
}

int launch_gemm_i8(cudaStream_t st, bool mn, const CUtensorMap* tmA, const CUtensorMap* tmB, double* out, int nrows, int kdim,
                   int S, int klen, int H, const int* rowexp, const int* rowbad, const int* colexp, int cstride, size_t slab,
                   size_t rs, size_t hs, const Scalars* sc, int num_sms) {
    if (H > 64) { set_error("H = %d > 64 is not supported by the INT8 contraction", H); return -1; }
    if (klen % KB != 0) { set_error("INT8 split-K chunk %d is not a multiple of %d", klen, KB); return -1; }
    if (nrows <= 0 || kdim <= 0 || H <= 0) return 0;
    const int nwork = ((nrows + TM - 1) / TM) * S;
    const int grid = std::max(1, std::min(nwork, num_sms));
    if (mn) gemm_i8_kernel<true><<<grid, 192, SMEM, st>>>(*tmA, *tmB, out, nrows, kdim, S, klen, H, i8_hpad(H), rowexp, rowbad, colexp, cstride, slab, rs, hs, sc);
    else gemm_i8_kernel<false><<<grid, 192, SMEM, st>>>(*tmA, *tmB, out, nrows, kdim, S, klen, H, i8_hpad(H), rowexp, rowbad, colexp, cstride, slab, rs, hs, sc);
    VB_LAUNCH_OK();
    return 0;
}

}  // namespace vb
