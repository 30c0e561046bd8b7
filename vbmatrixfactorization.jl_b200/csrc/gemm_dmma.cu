// K1 / K2: the two dense contractions over Y of one VB iteration, as TMA-fed FP64 tensor-core GEMMs.
//
//   K1  P = Y' * BHat   (M x H, K = L)    reference: src/vbmf.jl:98, src/vbmf_sparse.jl:195,232, src/vbmf_dual.jl:235,272
//   K2  Q = Y  * AHat   (L x H, K = M)    reference: src/vbmf.jl:112, src/vbmf_sparse.jl:266,317, src/vbmf_dual.jl:304,380
//
// sm_100a facts this design rests on (measured, profiles/r01_fp64_peak_microbench.jsonl): the FP64 tensor path is
// mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4 (tcgen05 has no f64 kind), one DMMA per 16 clk per SM sub-partition,
// 37.0 TFLOP/s chip-wide, dependent-issue latency ~26 clk (>= 2 independent accumulators per warp saturate it).
//
// Pipeline: one producer warp issues cp.async.bulk.tensor (TMA, SWIZZLE_128B) into a multi-stage shared-memory
// ring guarded by full/empty mbarriers; consumer warps read fragments with conflict-free 64-bit LDS and issue
// DMMA into register accumulators.  Persistent CTAs walk a static tile list.
//
// Bank-conflict-free fragment reads: every shared tile row is 128 B (16 doubles) and TMA XORs the 16-byte chunk
// index with (row & 7).  A 64-bit LDS is served per half-warp, so the 16 lanes of a half-warp must hit 16
// distinct 8-byte slots of the 128-byte bank line:
//   K1 (both operands K-contiguous): rows = fragment row r = lane>>2, the 4 k-values of one DMMA are taken at
//       e = 2*sp + (j&1) + 8*(j>>1) (j = lane&3, sp = 0..3) -- a fixed permutation of k applied to both operands.
//   K2 (both operands K-strided: rows are k): the fragment row index r selects the element inside the row as
//       e = 8*((r>>1)&1) + 2*t + (r&1) in box (r>>2), t = tile index mod 4 -- a permutation of the M / N index that
//       the epilogue undoes when it stores the accumulators.
#include "gemm.cuh"
#include <cstdlib>
#include <algorithm>

namespace vb {

// ------------------------------------------------------------------------------------------- PTX wrappers
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
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// Hand a pipeline stage back to the TMA producer.  The stage was read through the generic proxy (LDS) and will be
// overwritten through the async proxy (TMA): that write-after-read crosses proxies, so every reading lane issues
// fence.proxy.async before the release.  Without it a persistent CTA sporadically reads rows of the *next* k-block
// (observed on B200: a few rows per launch wrong once a CTA walks more than one tile; tools/k1race reproduces it).
__device__ __forceinline__ void consumer_release(uint32_t empty_bar, int lane) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_bar);
}
__device__ __forceinline__ double lds64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

constexpr int BM = 128;      // CTA tile rows (columns of Y in K1, rows of Y in K2)
constexpr int BK = 16;       // k extent of one pipeline stage = one 128-byte swizzle row
constexpr int BOX = BK * 16 * 8;  // bytes of one 16 x 16 box (K2)

template <int BN> struct Cfg;
template <> struct Cfg<32>  { static constexpr int WM = 4, WN = 1, STAGES = 5, CPS = 2; };
template <> struct Cfg<64>  { static constexpr int WM = 4, WN = 2, STAGES = 8, CPS = 1; };
template <> struct Cfg<128> { static constexpr int WM = 4, WN = 4, STAGES = 6, CPS = 1; };

// K1 has no constraint on the warp tile (its operand permutation is along k), so it can run more, smaller warp tiles:
// 4 consumer warps per sub-partition hide the LDS / mbarrier latency better (measured: 36.1 TFLOP/s for the 16-warp BN=128
// configuration against 34.8 for 8 warps at BN=64).  K2 needs 32 x 32 warp tiles (MT, NT multiples of 4).
#ifndef K1_WM64
#define K1_WM64 8
#endif
#ifndef K1_WM32
#define K1_WM32 8
#endif
template <int BN> struct CfgK1;
template <> struct CfgK1<32>  { static constexpr int WM = K1_WM32, WN = 1, STAGES = 5, CPS = 2; };
template <> struct CfgK1<64>  { static constexpr int WM = K1_WM64, WN = 2, STAGES = 8, CPS = 1; };
template <> struct CfgK1<128> { static constexpr int WM = 4, WN = 4, STAGES = 6, CPS = 1; };

template <int BN> struct Sizes {
    static constexpr int STAGE = (BM + BN) * BK * 8;
    static constexpr int SMEM = Cfg<BN>::STAGES * STAGE + 2 * Cfg<BN>::STAGES * 8 + 1024;
};

// ------------------------------------------------------------------------------------------- K1
template <int BN>
__global__ void __launch_bounds__((CfgK1<BN>::WM * CfgK1<BN>::WN + 1) * 32, CfgK1<BN>::CPS)
gemm_ytb_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmB,
                double* __restrict__ P, int M, int L, int H, int ldP, int S, int kb_per_split, size_t slab_stride,
                const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    constexpr int WM = CfgK1<BN>::WM, WN = CfgK1<BN>::WN, STAGES = CfgK1<BN>::STAGES;
    constexpr int NCW = WM * WN;
    constexpr int MT = BM / WM / 8, NT = BN / WN / 8;
    constexpr int YB = BM * BK * 8, SB = Sizes<BN>::STAGE;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t full0 = base + STAGES * SB, empty0 = full0 + STAGES * 8;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, NCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    // work item w = (m-tile, k-split): split-K over L evens out the tile count over the SMs (196 tiles on 148 SMs at
    // 25000 columns per GPU would otherwise cost two full rounds); the S slabs are summed in fixed order afterwards.
    const int nwork = ((M + BM - 1) / BM) * S;
    const int nkb = (L + BK - 1) / BK;

    if (warp == NCW) {  // ---------------- producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int m0 = (w / S) * BM, ks = w % S;
                const int kb0 = ks * kb_per_split, kb1 = min(nkb, kb0 + kb_per_split);
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    mbar_expect_tx(full0 + 8 * s, SB);
                    tma_load_2d(base + s * SB, &tmY, full0 + 8 * s, kb * BK, m0);
                    tma_load_2d(base + s * SB + YB, &tmB, full0 + 8 * s, kb * BK, 0);
                }
            }
        }
        return;
    }
    // ---------------- consumers
    const int r = lane >> 2, j = lane & 3;
    const int wm0 = (warp / WN) * (MT * 8), wn0 = (warp % WN) * (NT * 8);
    uint32_t off[4];
#pragma unroll
    for (int sp = 0; sp < 4; ++sp) off[sp] = r * 128 + (((sp + 4 * (j >> 1)) ^ r) << 4) + ((j & 1) << 3);

    uint32_t it = 0;
    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int tile = w / S, ks = w % S;
        const int kb0 = ks * kb_per_split, kb1 = min(nkb, kb0 + kb_per_split);
        double acc[MT][NT][2];
#pragma unroll
        for (int a = 0; a < MT; ++a)
#pragma unroll
            for (int b = 0; b < NT; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }

        for (int kb = kb0; kb < kb1; ++kb, ++it) {
            const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
            mbar_wait(full0 + 8 * s, ph);
            const uint32_t ys = base + s * SB + wm0 * 128, bs = base + s * SB + YB + wn0 * 128;
#pragma unroll
            for (int sp = 0; sp < 4; ++sp) {
                double af[MT], bf[NT];
#pragma unroll
                for (int a = 0; a < MT; ++a) af[a] = lds64(ys + a * 1024 + off[sp]);
#pragma unroll
                for (int b = 0; b < NT; ++b) bf[b] = lds64(bs + b * 1024 + off[sp]);
#pragma unroll
                for (int a = 0; a < MT; ++a)
#pragma unroll
                    for (int b = 0; b < NT; ++b) dmma(acc[a][b], af[a], bf[b]);
            }
            consumer_release(empty0 + 8 * s, lane);
        }
        // epilogue: raw P tile, row-major [M][ldP]
        const int m0 = tile * BM + wm0;
#pragma unroll
        for (int a = 0; a < MT; ++a) {
            const int m = m0 + a * 8 + r;
            if (m < M) {
#pragma unroll
                for (int b = 0; b < NT; ++b) {
                    const int h = wn0 + b * 8 + 2 * j;
                    double* p = P + (size_t)ks * slab_stride + (size_t)m * ldP + h;
                    if (h < H) p[0] = acc[a][b][0];
                    if (h + 1 < H) p[1] = acc[a][b][1];
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------- K2
// permuted index of fragment row/col q (0..7) of tile t (0..3) inside a 32-wide group
__device__ __forceinline__ int perm32(int q, int t) { return 16 * (q >> 2) + 8 * ((q >> 1) & 1) + 2 * t + (q & 1); }

template <int BN>
__global__ void __launch_bounds__((Cfg<BN>::WM * Cfg<BN>::WN + 1) * 32, Cfg<BN>::CPS)
gemm_ya_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmA,
               double* __restrict__ Qpart, int L, int M, int H, int ldQ, int kchunk, int S,
               const Scalars* __restrict__ sc) {
    if (sc != nullptr && !sc->active) return;
    constexpr int WM = Cfg<BN>::WM, WN = Cfg<BN>::WN, STAGES = Cfg<BN>::STAGES;
    constexpr int NCW = WM * WN;
    constexpr int MT = BM / WM / 8, NT = BN / WN / 8;
    static_assert(MT % 4 == 0 && NT % 4 == 0, "K2 needs 32-wide warp tiles");
    constexpr int YB = BM * BK * 8, SB = Sizes<BN>::STAGE;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t full0 = base + STAGES * SB, empty0 = full0 + STAGES * 8;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, NCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    const int ntl = (L + BM - 1) / BM;
    const int nwork = ntl * S;

    if (warp == NCW) {  // ---------------- producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int kc = w / ntl, l0 = (w % ntl) * BM;
                const int k_begin = kc * kchunk, k_end = min(M, k_begin + kchunk);
                for (int k = k_begin; k < k_end; k += BK, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    mbar_expect_tx(full0 + 8 * s, SB);
                    const uint32_t dst = base + s * SB;
#pragma unroll
                    for (int b = 0; b < BM / 16; ++b) tma_load_2d(dst + b * BOX, &tmY, full0 + 8 * s, l0 + 16 * b, k);
#pragma unroll
                    for (int b = 0; b < BN / 16; ++b) tma_load_2d(dst + YB + b * BOX, &tmA, full0 + 8 * s, 16 * b, k);
                }
            }
        }
        return;
    }
    // ---------------- consumers
    const int r = lane >> 2, j = lane & 3;
    const int wl0 = (warp / WN) * (MT * 8), wn0 = (warp % WN) * (NT * 8);
    const int chi = (r >> 1) & 1;
    // byte offset of this lane's element for k4-step sp and tile-in-group t, relative to the 32-wide group base
    const uint32_t rowoff = j * 128 + ((r & 1) << 3) + (r >> 2) * BOX;

    uint32_t it = 0;
    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int kc = w / ntl, l0 = (w % ntl) * BM;
        const int k_begin = kc * kchunk, k_end = min(M, k_begin + kchunk);
        double acc[MT][NT][2];
#pragma unroll
        for (int a = 0; a < MT; ++a)
#pragma unroll
            for (int b = 0; b < NT; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }

        for (int k = k_begin; k < k_end; k += BK, ++it) {
            const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
            mbar_wait(full0 + 8 * s, ph);
            const uint32_t ys = base + s * SB + (wl0 / 16) * BOX + rowoff;
            const uint32_t as = base + s * SB + YB + (wn0 / 16) * BOX + rowoff;
#pragma unroll
            for (int sp = 0; sp < 4; ++sp) {
                double af[MT], bf[NT];
                const uint32_t hi = (uint32_t)((chi ^ (sp & 1)) << 6) + sp * 512;
#pragma unroll
                for (int a = 0; a < MT; ++a) af[a] = lds64(ys + (a >> 2) * (2 * BOX) + hi + (((a & 3) ^ j) << 4));
#pragma unroll
                for (int b = 0; b < NT; ++b) bf[b] = lds64(as + (b >> 2) * (2 * BOX) + hi + (((b & 3) ^ j) << 4));
#pragma unroll
                for (int a = 0; a < MT; ++a)
#pragma unroll
                    for (int b = 0; b < NT; ++b) dmma(acc[a][b], af[a], bf[b]);
            }
            consumer_release(empty0 + 8 * s, lane);
        }
        // epilogue: undo the permutation, store the split-K slab column-major [H][ldQ]
        double* slab = Qpart + (size_t)kc * H * ldQ;
#pragma unroll
        for (int a = 0; a < MT; ++a) {
            const int l = l0 + wl0 + 32 * (a >> 2) + perm32(r, a & 3);
            if (l < L) {
#pragma unroll
                for (int b = 0; b < NT; ++b) {
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int h = wn0 + 32 * (b >> 2) + perm32(2 * j + i, b & 3);
                        if (h < H) slab[(size_t)h * ldQ + l] = acc[a][b][i];
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------- host side
static PFN_encodeTiled g_encode = nullptr;

PFN_encodeTiled tmap_encoder() {
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
            set_error("cuTensorMapEncodeTiled entry point not available (%s)", cudaGetErrorString(e));
            return nullptr;
        }
        g_encode = (PFN_encodeTiled)fn;
    }
    return g_encode;
}

int make_tmap_2d(CUtensorMap* out, const void* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_bytes,
                 uint32_t box0, uint32_t box1) {
    if (!tmap_encoder()) return -1;
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (stride1_bytes & 15) != 0) {
        set_error("TMA tensor map needs 16-byte aligned base and pitch (base=%p pitch=%llu)", base,
                  (unsigned long long)stride1_bytes);
        return -1;
    }
    cuuint64_t dims[2] = {dim0, dim1};
    cuuint64_t strides[1] = {stride1_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (dims %llu x %llu, pitch %llu, box %u x %u)", (int)r,
                  (unsigned long long)dim0, (unsigned long long)dim1, (unsigned long long)stride1_bytes, box0, box1);
        return -1;
    }
    return 0;
}

GemmGeometry gemm_geometry(int H) {
    GemmGeometry g;
    if (H <= 32) { g.bn = 32; g.ctas_per_sm = Cfg<32>::CPS; g.stages = Cfg<32>::STAGES; }
    else if (H <= 64) { g.bn = 64; g.ctas_per_sm = Cfg<64>::CPS; g.stages = Cfg<64>::STAGES; }
    else { g.bn = 128; g.ctas_per_sm = Cfg<128>::CPS; g.stages = Cfg<128>::STAGES; }
    return g;
}

void plan_splitk(int L, int M, int H, int num_sms, int* S_out, int* kchunk_out) {
    if (M <= 0 || L <= 0) { *S_out = 1; *kchunk_out = BK; return; }
    const GemmGeometry g = gemm_geometry(H);
    const long cap = (long)num_sms * g.ctas_per_sm;
    const long ntl = (L + BM - 1) / BM;
    const int ldq = (L + 1) & ~1;
    int best_s = 1;
    double best_eff = 0.0;
    for (int s = 1; s <= 256; ++s) {
        long kc = (((long)M + s - 1) / s + BK - 1) / BK * BK;
        if (kc < 512 && s > 1) break;                               // keep the main loop long enough to amortise fill/drain
        if ((long)s * H * ldq * 8 > (1L << 30) && s > 1) break;      // slab workspace cap: 1 GiB
        long s_eff = ((long)M + kc - 1) / kc;                        // slabs actually non-empty
        long work = ntl * s_eff;
        double eff = (double)work / (double)(((work + cap - 1) / cap) * cap);
        if (eff > best_eff + 0.01) { best_eff = eff; best_s = (int)s_eff; }
    }
    long kc = (((long)M + best_s - 1) / best_s + BK - 1) / BK * BK;
    if (kc < BK) kc = BK;
    *S_out = (int)(((long)M + kc - 1) / kc);
    if (*S_out < 1) *S_out = 1;
    *kchunk_out = (int)kc;
}

void plan_splitk_ytb(int L, int M, int H, int num_sms, int* S_out, int* kb_per_split) {
    const GemmGeometry g = gemm_geometry(H);
    const long cap = (long)num_sms * g.ctas_per_sm;
    const long ntiles = (M + BM - 1) / BM, nkb = (L + BK - 1) / BK;
    int best_s = 1;
    double best_eff = 0.0;
    for (int s = 1; s <= 16; ++s) {
        const long kbs = (nkb + s - 1) / s;
        if (kbs < 48 && s > 1) break;                      // keep >= 48 k-blocks per item (pipeline fill/drain, epilogue)
        const long s_eff = (nkb + kbs - 1) / kbs;
        const long work = ntiles * s_eff;
        // slab traffic (write + read of s partial outputs) relative to the Y bytes of the launch
        const double extra = s_eff > 1 ? 2.0 * s_eff * H / (double)L : 0.0;
        const double eff = (double)work / (double)(((work + cap - 1) / cap) * cap) / (1.0 + extra);
        if (eff > best_eff + 0.005) { best_eff = eff; best_s = (int)s_eff; }
    }
    const long kbs = (nkb + best_s - 1) / best_s;
    *S_out = (int)std::max<long>(1, (nkb + kbs - 1) / std::max<long>(kbs, 1));
    *kb_per_split = (int)std::max<long>(kbs, 1);
}

template <int BN>
static int launch_ytb_t(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmB, double* P, int M, int L, int H,
                        int ldP, int S, int kbs, size_t slab_stride, const Scalars* sc, int num_sms) {
    const int nwork = ((M + BM - 1) / BM) * S;
    const int grid = std::max(1, std::min(nwork, num_sms * CfgK1<BN>::CPS));
    const int threads = (CfgK1<BN>::WM * CfgK1<BN>::WN + 1) * 32;
    gemm_ytb_kernel<BN><<<grid, threads, Sizes<BN>::SMEM, st>>>(*tmY, *tmB, P, M, L, H, ldP, S, kbs, slab_stride, sc);
    VB_LAUNCH_OK();
    return 0;
}

// cudaFuncSetAttribute is per device: called once per context for the context's device (no process-wide flags)
int gemm_init_device() {
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ytb_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<32>::SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ytb_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<64>::SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ytb_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<128>::SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ya_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<32>::SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ya_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<64>::SMEM));
    VB_CUDA_OK(cudaFuncSetAttribute(gemm_ya_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sizes<128>::SMEM));
    return gemm_i8_init_device();
}

int launch_gemm_ytb(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmB, double* P, int M, int L, int H,
                    int ldP, int S, int kb_per_split, size_t slab_stride, const Scalars* sc, int num_sms) {
    if (H > 128) { set_error("H = %d > 128 is not supported by the K1 kernel yet", H); return -1; }
    if (M <= 0 || L <= 0 || H <= 0) return 0;
    if (H <= 32) return launch_ytb_t<32>(st, tmY, tmB, P, M, L, H, ldP, S, kb_per_split, slab_stride, sc, num_sms);
    if (H <= 64) return launch_ytb_t<64>(st, tmY, tmB, P, M, L, H, ldP, S, kb_per_split, slab_stride, sc, num_sms);
    return launch_ytb_t<128>(st, tmY, tmB, P, M, L, H, ldP, S, kb_per_split, slab_stride, sc, num_sms);
}

template <int BN>
static int launch_ya_t(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmA, double* Qpart, int L, int M, int H,
                       int ldQ, int kchunk, int S, const Scalars* sc, int num_sms) {
    const int ntl = (L + BM - 1) / BM;
    const int grid = std::max(1, std::min(ntl * S, num_sms * Cfg<BN>::CPS));
    const int threads = (Cfg<BN>::WM * Cfg<BN>::WN + 1) * 32;
    gemm_ya_kernel<BN><<<grid, threads, Sizes<BN>::SMEM, st>>>(*tmY, *tmA, Qpart, L, M, H, ldQ, kchunk, S, sc);
    VB_LAUNCH_OK();
    return 0;
}

int launch_gemm_ya(cudaStream_t st, const CUtensorMap* tmY, const CUtensorMap* tmA, double* Qpart, int L, int M, int H,
                   int ldQ, int kchunk, int S, const Scalars* sc, int num_sms) {
    if (H > 128) { set_error("H = %d > 128 is not supported by the K2 kernel yet", H); return -1; }
    if (M <= 0 || L <= 0 || H <= 0) return 0;
    if (kchunk % BK != 0) { set_error("split-K chunk %d is not a multiple of %d", kchunk, BK); return -1; }
    if (H <= 32) return launch_ya_t<32>(st, tmY, tmA, Qpart, L, M, H, ldQ, kchunk, S, sc, num_sms);
    if (H <= 64) return launch_ya_t<64>(st, tmY, tmA, Qpart, L, M, H, ldQ, kchunk, S, sc, num_sms);
    return launch_ya_t<128>(st, tmY, tmA, Qpart, L, M, H, ldQ, kchunk, S, sc, num_sms);
}

// ------------------------------------------------------------------------------------------- SIMT cross-check kernels
__global__ void gemm_ytb_simt_kernel(const double* __restrict__ Y, int ldY, const double* __restrict__ B, int ldB,
                                     double* __restrict__ P, int M, int L, int H, int ldP, const Scalars* sc) {
    if (sc != nullptr && !sc->active) return;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long)M * H) return;
    const int m = (int)(idx / H), h = (int)(idx % H);
    const double* y = Y + (size_t)m * ldY;
    const double* b = B + (size_t)h * ldB;
    double s = 0.0;
    for (int l = 0; l < L; ++l) s = fma(y[l], b[l], s);
    P[(size_t)m * ldP + h] = s;
}

__global__ void gemm_ya_simt_kernel(const double* __restrict__ Y, int ldY, const double* __restrict__ A,
                                    double* __restrict__ Qpart, int L, int M, int H, int ldQ, int kchunk, int S,
                                    const Scalars* sc) {
    if (sc != nullptr && !sc->active) return;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long)S * H * L) return;
    const int l = (int)(idx % L);
    const int h = (int)((idx / L) % H);
    const int kc = (int)(idx / ((long)L * H));
    const int k_begin = kc * kchunk, k_end = min(M, k_begin + kchunk);
    double s = 0.0;
    for (int m = k_begin; m < k_end; ++m) s = fma(Y[(size_t)m * ldY + l], A[(size_t)m * H + h], s);
    Qpart[(size_t)kc * H * ldQ + (size_t)h * ldQ + l] = s;
}

int launch_gemm_ytb_simt(cudaStream_t st, const double* Y, int ldY, const double* B, int ldB, double* P, int M, int L,
                         int H, int ldP, const Scalars* sc) {
    const long n = (long)M * H;
    if (n <= 0) return 0;
    gemm_ytb_simt_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Y, ldY, B, ldB, P, M, L, H, ldP, sc);
    VB_LAUNCH_OK();
    return 0;
}

int launch_gemm_ya_simt(cudaStream_t st, const double* Y, int ldY, const double* A, double* Qpart, int L, int M, int H,
                        int ldQ, int kchunk, int S, const Scalars* sc) {
    const long n = (long)S * H * L;
    if (n <= 0) return 0;
    gemm_ya_simt_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Y, ldY, A, Qpart, L, M, H, ldQ, kchunk, S, sc);
    VB_LAUNCH_OK();
    return 0;
}

}  // namespace vb
