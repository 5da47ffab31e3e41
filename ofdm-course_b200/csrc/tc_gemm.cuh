// tcgen05 building blocks for the batched OMP correlation (sm_100a): TMA-fed shared-memory ring, single-thread
// tcgen05.mma (kind::tf32, FP32 accumulators in TMEM), tcgen05.ld epilogue.  Hand-written PTX; the descriptor bit
// layouts follow the PTX ISA "tcgen05 matrix / instruction descriptor" tables.
//   D[M x N] (+)= A[M x K] * B[N x K]^T     A, B: FP32 storage, K-major (K contiguous), consumed as TF32.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define TC_BM 128                    // rows of A per CTA = TMEM lanes
#define TC_BN 128                    // rows of B per tile = TMEM columns (FP32)
#define TC_BK 32                     // TF32 elements per k-block: 128 bytes = one 128B-swizzle span
#define TC_UK 8                      // K per tcgen05.mma for kind::tf32
#define TC_STAGES 4
#define TC_THREADS 192               // warp 0: TMA producer, warp 1: TMEM owner + MMA issuer, warps 2..5: epilogue
#define TC_TILE_A_BYTES (TC_BM * TC_BK * 4)
#define TC_TILE_B_BYTES (TC_BN * TC_BK * 4)
#define TC_STAGE_BYTES (TC_TILE_A_BYTES + TC_TILE_B_BYTES)
#define TC_SMEM_BYTES (TC_STAGES * TC_STAGE_BYTES + 1024 + 256)

// ---------------------------------------------------------------- host: tensor maps
typedef CUresult (*tc_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// The lookup runs once, under the C++ guarantee for function-local statics, so contexts on several host threads
// (ofdm_group) never race on it.
static inline tc_encode_fn tc_get_encode() {
    static const tc_encode_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return (tc_encode_fn)p;
        return (tc_encode_fn) nullptr;
    }();
    return fn;
}
// rows x K FP32 matrix, K contiguous; box = 128 rows x 32 floats (128 B), 128B swizzle
// `ld` (elements, 0 = K): row pitch when the K extent addressed is a slice of wider rows
static inline bool tc_make_kmajor_map(CUtensorMap* map, const void* base, uint64_t rows, uint64_t K, uint64_t ld = 0) {
    tc_encode_fn enc = tc_get_encode();
    if (!enc) return false;
    cuuint64_t dims[2] = {K, rows};
    cuuint64_t strides[1] = {(ld ? ld : K) * sizeof(float)};
    cuuint32_t box[2] = {TC_BK, 128};
    cuuint32_t estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---------------------------------------------------------------- device: PTX wrappers
__device__ __forceinline__ uint32_t tc_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem(bar)), "r"(count)); }
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem(bar)) : "memory"); }
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "TCW_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TCD_%=;\n\t"
        "bra TCW_%=;\n\t"
        "TCD_%=:\n\t}" ::"r"(tc_smem(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_tma_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(tc_smem(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(tc_smem(bar))
                 : "memory");
}
// shared-memory matrix descriptor: K-major, 128B swizzle, 8-row groups 1024 B apart (SBO), descriptor version 1
__device__ __forceinline__ uint64_t tc_desc_kmajor_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128, N = TC_BN
#define TC_IDESC ((1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24))
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_tmem_dealloc(uint32_t base, uint32_t ncols) {     // whole warp, the allocating one
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
// 32 lanes x 32 consecutive FP32 columns -> 32 registers per thread (lane i of the warp reads TMEM lane base_lane + i)
__device__ __forceinline__ void tc_tmem_ld32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
          "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

struct TcShared {
    uint64_t full[TC_STAGES], empty[TC_STAGES], tmem_full;
    uint32_t tmem_base;
};

// Mainloop of one 128 x 128 output tile: producer and MMA roles.  `tiles` = 1024-aligned stage ring.
// Called by warps 0 and 1; returns when every k-block has been issued (MMA warp has committed tmem_full).
__device__ __forceinline__ void tc_mainloop(TcShared* sh, unsigned char* tiles, const CUtensorMap* mapA, const CUtensorMap* mapB, int m0, int n0, int nkb,
                                            uint32_t tmem_d, int warp, int lane, uint32_t& it) {
    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % TC_STAGES;
                tc_mbar_wait(&sh->empty[s], ((it / TC_STAGES) & 1) ^ 1);
                tc_mbar_expect_tx(&sh->full[s], TC_STAGE_BYTES);
                unsigned char* a = tiles + s * TC_STAGE_BYTES;
                tc_tma_2d(a, mapA, kb * TC_BK, m0, &sh->full[s]);
                tc_tma_2d(a + TC_TILE_A_BYTES, mapB, kb * TC_BK, n0, &sh->full[s]);
            }
        } else it += nkb;
        it = __shfl_sync(0xffffffffu, it, 0);
    } else if (warp == 1) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % TC_STAGES;
                tc_mbar_wait(&sh->full[s], (it / TC_STAGES) & 1);
                tc_fence_after();
                const uint32_t a = tc_smem(tiles + s * TC_STAGE_BYTES);
                const uint64_t ad = tc_desc_kmajor_sw128(a), bd = tc_desc_kmajor_sw128(a + TC_TILE_A_BYTES);
#pragma unroll
                for (int k = 0; k < TC_BK / TC_UK; ++k)   // advance 32 bytes (>>4 = 2) inside the 128-byte swizzle span
                    tc_mma_tf32(tmem_d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), TC_IDESC, (kb | k) ? 1u : 0u);
                tc_commit(&sh->empty[s]);                  // frees the stage when these MMAs have read it
            }
            tc_commit(&sh->tmem_full);                     // accumulator complete
        } else it += nkb;
        it = __shfl_sync(0xffffffffu, it, 0);
    }
}

// Bring-up kernel: one tile per CTA, accumulator written to global memory.
static __global__ void __launch_bounds__(TC_THREADS) tc_gemm_store_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                                   float* __restrict__ D, int ldd, int K, int n_fastest) {
    extern __shared__ unsigned char tc_smem_raw[];
    unsigned char* tiles = (unsigned char*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
    TcShared* sh = (TcShared*)(tiles + TC_STAGES * TC_STAGE_BYTES);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // n_fastest: consecutive CTAs walk the N tiles of ONE row block (they share the A tile through L2); else the M tiles
    const int m0 = (n_fastest ? blockIdx.y : blockIdx.x) * TC_BM, n0 = (n_fastest ? blockIdx.x : blockIdx.y) * TC_BN;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { tc_mbar_init(&sh->full[s], 1); tc_mbar_init(&sh->empty[s], 1); }
        tc_mbar_init(&sh->tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tc_tmem_alloc(&sh->tmem_base, TC_BN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = sh->tmem_base;
    uint32_t it = 0;
    if (warp < 2) {
        tc_mainloop(sh, tiles, &mapA, &mapB, m0, n0, K / TC_BK, tmem_d, warp, lane, it);
    } else {
        tc_mbar_wait(&sh->tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3;                              // TMEM lane quarter this warp may access
        const int row = m0 + 32 * q + lane;
        float v[32];
#pragma unroll 1
        for (int c0 = 0; c0 < TC_BN; c0 += 32) {
            tc_tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) D[(size_t)row * ldd + n0 + c0 + j] = v[j];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tc_tmem_dealloc(tmem_d, TC_BN);
}

// ---------------------------------------------------------------------------------------------------------
// Batched OMP correlation with a fused arg-top epilogue.
//   A operand  Rt [frames_pad x K2]   row f = [Re r_f | Im r_f]                       (K2 = 2*Np padded to 32)
//   B operand  Bt [2*L_pad x K2]      row 2l = [Re a_l | Im a_l], row 2l+1 = [-Im a_l | Re a_l]
//   => D[f][2l] = Re(a_l^H r_f), D[f][2l+1] = Im(a_l^H r_f): frames on TMEM lanes, dictionary along columns, so
// each epilogue thread owns one frame and keeps its TC_TOP best |a_l^H r|^2 locally; the 2*L x frames
// correlation matrix never leaves the SM.  TF32 scores only *screen*: the caller re-scores the candidates in FP32.
// One CTA = 128 frames, persistent over all dictionary tiles; two TMEM accumulators (2 x 128 columns) let the
// epilogue of tile t overlap the MMAs of tile t+1.
// ---------------------------------------------------------------------------------------------------------
#define TC_TOP 4
struct TcSharedTop {
    uint64_t full[TC_STAGES], empty[TC_STAGES], tfull[2], tempty[2];
    uint32_t tmem_base;
};
#define TC_SMEM_TOP_BYTES (TC_STAGES * TC_STAGE_BYTES + 1024 + 256)

static __global__ void __launch_bounds__(TC_THREADS) tc_corr_top_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, int ntiles,
                                                                 int K2, int Ldict, int32_t* __restrict__ cand, float* __restrict__ cand_score) {
    extern __shared__ unsigned char tc_smem_raw[];
    unsigned char* tiles = (unsigned char*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
    TcSharedTop* sh = (TcSharedTop*)(tiles + TC_STAGES * TC_STAGE_BYTES);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * TC_BM;
    const int nkb = K2 / TC_BK;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { tc_mbar_init(&sh->full[s], 1); tc_mbar_init(&sh->empty[s], 1); }
        for (int b = 0; b < 2; ++b) { tc_mbar_init(&sh->tfull[b], 1); tc_mbar_init(&sh->tempty[b], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tc_tmem_alloc(&sh->tmem_base, 2 * TC_BN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = sh->tmem_base;
    if (warp == 0) {
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = 0; t < ntiles; ++t)
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % TC_STAGES;
                    tc_mbar_wait(&sh->empty[s], ((it / TC_STAGES) & 1) ^ 1);
                    tc_mbar_expect_tx(&sh->full[s], TC_STAGE_BYTES);
                    unsigned char* a = tiles + s * TC_STAGE_BYTES;
                    tc_tma_2d(a, &mapA, kb * TC_BK, m0, &sh->full[s]);
                    tc_tma_2d(a + TC_TILE_A_BYTES, &mapB, kb * TC_BK, t * TC_BN, &sh->full[s]);
                }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = 0; t < ntiles; ++t) {
                const int buf = t & 1;
                tc_mbar_wait(&sh->tempty[buf], ((t >> 1) & 1) ^ 1);      // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t td = tmem_d + buf * TC_BN;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % TC_STAGES;
                    tc_mbar_wait(&sh->full[s], (it / TC_STAGES) & 1);
                    tc_fence_after();
                    const uint32_t a = tc_smem(tiles + s * TC_STAGE_BYTES);
                    const uint64_t ad = tc_desc_kmajor_sw128(a), bd = tc_desc_kmajor_sw128(a + TC_TILE_A_BYTES);
#pragma unroll
                    for (int k = 0; k < TC_BK / TC_UK; ++k) tc_mma_tf32(td, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), TC_IDESC, (kb | k) ? 1u : 0u);
                    tc_commit(&sh->empty[s]);
                }
                tc_commit(&sh->tfull[buf]);
            }
        }
    } else {
        const int q = warp & 3;
        float best[TC_TOP];
        int bidx[TC_TOP];
#pragma unroll
        for (int i = 0; i < TC_TOP; ++i) { best[i] = -1.f; bidx[i] = 0; }
        float v[32];
        for (int t = 0; t < ntiles; ++t) {
            const int buf = t & 1;
            tc_mbar_wait(&sh->tfull[buf], (t >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int c0 = 0; c0 < TC_BN; c0 += 32) {
                tc_tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + buf * TC_BN + c0, v);
                const int l0 = (t * TC_BN + c0) >> 1;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float sc = v[2 * j] * v[2 * j] + v[2 * j + 1] * v[2 * j + 1];
                    const int l = l0 + j;
                    if (sc > best[TC_TOP - 1] && l < Ldict) {          // insertion into the sorted top list (rare)
                        best[TC_TOP - 1] = sc; bidx[TC_TOP - 1] = l;
#pragma unroll
                        for (int i = TC_TOP - 1; i > 0; --i)
                            if (best[i] > best[i - 1]) { float ts = best[i]; best[i] = best[i - 1]; best[i - 1] = ts; int ti = bidx[i]; bidx[i] = bidx[i - 1]; bidx[i - 1] = ti; }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) tc_mbar_arrive(&sh->tempty[buf]);
        }
        const int64_t f = m0 + 32 * q + lane;
#pragma unroll
        for (int i = 0; i < TC_TOP; ++i) { cand[f * TC_TOP + i] = bidx[i]; cand_score[f * TC_TOP + i] = best[i]; }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tc_tmem_dealloc(tmem_d, 2 * TC_BN);
}
