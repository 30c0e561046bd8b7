// Launcher interface of the two FP64 tensor-core (DMMA) contractions of the VB loop.
#pragma once
#include "common.cuh"

namespace vb {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// cuTensorMapEncodeTiled from the driver (nullptr and an error message when it is missing)
PFN_encodeTiled tmap_encoder();

// Encode a rank-2 FP64 tensor map (dim0 contiguous) with 128-byte swizzle and zero OOB fill.
int make_tmap_2d(CUtensorMap* out, const void* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_bytes,
                 uint32_t box0, uint32_t box1);

struct GemmGeometry {
    int bn;          // N tile (32 / 64 / 128), smallest >= H
    int ctas_per_sm;
    int stages;
};
GemmGeometry gemm_geometry(int H);
// opt the contraction kernels into their dynamic shared memory on the CURRENT device (once per context)
int gemm_init_device();

// K1: P[m][h] = sum_l Y[l, m] * B[l, h]      (Y' * BHat, src/vbmf.jl:98, src/vbmf_sparse.jl:195,232)
// tmY : dims {L, M}, box {16, 128};  tmB : dims {L, H} (column h contiguous in l), box {16, bn}
// P is row-major [M][ldP].
// With S > 1 the kernel writes S slabs P + s*slab_stride (split over L, kb_per_split 16-row blocks each) that the caller
// sums in fixed order (deterministic split-K); S == 1 writes P directly.
int launch_gemm_ytb(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmB, double* P,
                    int M, int L, int H, int ldP, int S, int kb_per_split, size_t slab_stride, const Scalars* sc, int num_sms);
void plan_splitk_ytb(int L, int M, int H, int num_sms, int* S, int* kb_per_split);

// K2: Qpart[s][h][l] = sum_{m in chunk s} Y[l, m] * A[m][h]   (Y * AHat, src/vbmf.jl:112, src/vbmf_sparse.jl:266)
// tmY : dims {L, M}, box {16, 16};  tmA : dims {H, M} (row m contiguous in h), box {16, 16}
// Qpart is S slabs of column-major [H][ldQ]; the caller reduces the slabs in fixed order (deterministic split-K).
int launch_gemm_ya(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmA, double* Qpart,
                   int L, int M, int H, int ldQ, int kchunk, int S, const Scalars* sc, int num_sms);

// split-K plan for K2: number of slabs and chunk length (multiple of 16)
void plan_splitk(int L, int M, int H, int num_sms, int* S, int* kchunk);

// ---- INT8 tensor-core contractions with exact slice splitting (gemm_int8.cu), H <= 64 ----
// Operands are I8_NSL signed radix-256 digit planes, int8 [I8_NSL][rows][ld], ld a multiple of 16; exponents are ints (2^e
// scales).
constexpr int I8_NSL = 7;
inline int i8_hpad(int H) { return (H + 15) / 16 * 16; }
inline int i8_ld(int n) { return (n + 15) / 16 * 16; }
int gemm_i8_init_device();
// rank-3 uint8 tensor map {d0, d1, d2} with byte pitches s1, s2; 32-byte swizzle, or 128-byte with swizzle128
int make_tmap_3d_i8(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2,
                    uint32_t b0, uint32_t b1, uint32_t b2, bool swizzle128);
// Y (L x M, column-major) -> row exponents F[L], column exponents E[M] (both over the finite values), digits Z [7][M][ldZ]
// (ldZ = i8_ld(L)), and the flags Fbad[L] / Ebad[M]: row / column holds a NaN or Inf
int i8_build_Y(cudaStream_t st, const double* Y, int ldY, int L, int M, uint8_t* Z, int ldZ, int* F, int* E, int* Fbad, int* Ebad);
// K1 operand: diag(2^F) * B (B column-major [H][ldB]) -> exponents G[Hp], digits W [7][Hp][ldZ]
int i8_slice_B(cudaStream_t st, const double* B, int ldB, int L, int H, const int* F, uint8_t* W, int ldZ, int* G, const Scalars* sc);
// K2 operand: diag(2^E) * A (A row-major [M][H]) -> exponents G[S][Hp] per split-K chunk of kchunk rows, digits W [7][Hp][ldM]
int i8_slice_A(cudaStream_t st, const double* A, int M, int H, const int* E, int kchunk, int S, uint8_t* W, int ldM, int* G, const Scalars* sc);
// out[s*slab + row*rs + h*hs] = 2^(rowexp[row] + colexp[s*cstride + h]) * sum_{k in split s} A(row, k) * B(k, h), NaN where
// rowbad[row] != 0 or the operand column held a NaN or Inf (non-finite inputs give NaN, never a finite value).
// mn = false (K1): tmA = Y digits {L, M, 7}, box {32, 128, 7}, 32-byte swizzle; rows are columns of Y, k = l.
// mn = true  (K2): tmA = Y digits {L, M, 7}, box {128, 32, 7}, 128-byte swizzle; rows are rows of Y, k = m.
// tmB: operand digits {kdim, Hp, 7}, box {32, Hp, 7}, 32-byte swizzle.  klen: split length, a multiple of 32.
int launch_gemm_i8(cudaStream_t st, bool mn, const CUtensorMap* tmA, const CUtensorMap* tmB, double* out, int nrows, int kdim,
                   int S, int klen, int H, const int* rowexp, const int* rowbad, const int* colexp, int cstride, size_t slab,
                   size_t rs, size_t hs, const Scalars* sc, int num_sms);

// Plain SIMT FP64 versions (debug / cross-check only; selected with VBMF_B200_GEMM=simt).
int launch_gemm_ytb_simt(cudaStream_t st, const double* Y, int ldY, const double* B, int ldB, double* P,
                         int M, int L, int H, int ldP, const Scalars* sc);
int launch_gemm_ya_simt(cudaStream_t st, const double* Y, int ldY, const double* A, double* Qpart,
                        int L, int M, int H, int ldQ, int kchunk, int S, const Scalars* sc);

}  // namespace vb
