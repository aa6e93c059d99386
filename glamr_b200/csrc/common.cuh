// Shared device/host helpers for the glamr_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/glamr_b200.h"

#define GLAMR_CUDA_TRY(expr)                       \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

#define GLAMR_LAUNCH_CHECK()                       \
  do {                                             \
    cudaError_t _e = cudaGetLastError();           \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

// Work-skipping experiment switches (tools/*_exp.py) exist only in a -DGLAMR_EXPERIMENT build; the release library that
// bench.py and the tests load has them compiled out.
#ifdef GLAMR_EXPERIMENT
#define GLAMR_DBG(x) (x)
#else
#define GLAMR_DBG(x) 0
#endif

// Which implementation runs when the environment does not say otherwise.  A path becomes the default only after its parity
// tests passed on a B200 (GLAMR_LBS_PATH=tc|tcblend|simt selects explicitly for A/B runs).
#define GLAMR_DEFAULT_LBS_TC 2        /* 2 = tensor-core blend + tensor-core skinning (verified on B200: all GPU tests green, memcheck clean), 1 = tensor-core blend + SIMT skinning, 0 = FP32 SIMT kernel */
#define GLAMR_DEFAULT_NET_WIMG 0       /* prior-network GEMMs: weight operand as a pre-split image fetched by bulk TMA (GLAMR_NET_WIMG=1) */

namespace glamr {

constexpr int kV = GLAMR_NUM_VERTS;          // 6890
constexpr int kNJ = GLAMR_NUM_JOINTS;        // 24
constexpr int kNB = GLAMR_NUM_BETAS;         // 10
constexpr int kPF = GLAMR_NUM_POSE_FEAT;     // 207
constexpr int kPFPad = 208;                  // row stride of the pose-feature scratch
constexpr int kVTile = 128;                  // vertices per LBS CTA
constexpr int kNVTiles = (kV + kVTile - 1) / kVTile;   // 54
constexpr int kVPad = kNVTiles * kVTile;     // 6912
constexpr int kTileCols = kVTile * 3;        // 384 posedirs columns per tile
constexpr int kChunkK = 9;                   // pose-feature rows per pipeline stage (= one joint's 3x3)
constexpr int kNChunks = kPF / kChunkK;      // 23
// tensor-core blend GEMM  v_posed[frame, col] = sum_k feat[frame, k] * basis[col, k]  (smpl_kernels.cu, lbs_blend_tc_kernel):
// k = 0..206 pose feature x posedirs, 207..216 betas x shapedirs, 217 = 1 x v_template, zero padded to 224
constexpr int kTcFeat = kPF + kNB + 1;       // 218
constexpr int kTcK = 224;                    // K padded to a multiple of the per-stage chunk
constexpr int kTcChunkK = 8;                 // one tcgen05 kind::tf32 MMA step per pipeline stage
constexpr int kTcChunks = kTcK / kTcChunkK;  // 28
constexpr int kTcM = 128;                    // frames per CTA tile (= TMEM lanes)
constexpr int kTcN = 256;                    // basis columns per CTA tile (= TMEM columns)
constexpr int kTcNTiles = (kV * 3 + kTcN - 1) / kTcN;   // 81
constexpr int kTcCols = kTcNTiles * kTcN;    // 20736
constexpr int kTcAStageFloats = 2 * (kTcChunkK / 4) * kTcM * 4;   // hi | lo images of a [128 x 8] K-major core-matrix tile: 2048 floats
constexpr int kTcBStageFloats = 2 * (kTcChunkK / 4) * kTcN * 4;   // 4096 floats
// tensor-core skinning (lbs_skin_tc_kernel): T[vertex][frame x 12] = W[vertex][24 joints] . A[24 joints][frame x 12]
constexpr int kSkF = 20;                     // frames per CTA tile
constexpr int kSkN = kSkF * 12;              // 240 TMEM columns: the 3x4 blended transform of each frame
constexpr int kSkKGroups = kNJ / 4;          // 6 groups of 4 joints (K = 24 = 3 MMA steps of 8)
constexpr int kSkWHalf = kSkKGroups * kVTile * 4;     // 3072 floats: hi (or lo) image of a [128 vertices x 24] K-major tile
constexpr int kSkWImageFloats = 2 * kSkWHalf;          // 6144 floats = 24,576 B per vertex tile
constexpr int kSkBHalf = kSkKGroups * kSkN * 4;        // 5760 floats: hi (or lo) image of a [240 x 24] K-major tile
constexpr int kSkBImageFloats = 2 * kSkBHalf;          // 11520 floats = 46,080 B per 20-frame tile
constexpr int kSkVpTileFloats = kTileCols * kSkF;      // 7680 floats = 30,720 B: v_posed of 128 vertices x 20 frames

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier + 1-D bulk TMA (cp.async.bulk) wrappers -------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// raise the pending transaction count without arriving (the arrival comes later with mbar_expect_tx)
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t addr = smem_u32(bar);
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
// global -> shared bulk copy through the TMA engine; completion is signalled on `bar` (complete_tx::bytes).
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- tcgen05 (UMMA) helpers: shared-memory descriptor of a K-major, un-swizzled operand tile and one kind::tf32 MMA ----
// rows = rows of the operand tile (128 for X, NT for W): fixes the leading byte offset between 16-byte K groups
__device__ __forceinline__ uint64_t umma_desc_kmajor_noswizzle(const void* smem_ptr, int rows) {
  // cute::UMMA::SmemDescriptor: start[0,14) | LBO[16,30) | SBO[32,46) | version=1 [46,48) | layout_type=0 [61,64)
  const uint32_t addr = smem_u32(smem_ptr);
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((rows * 16) >> 4) << 16;     // leading byte offset: next 16-byte K group
  d |= (uint64_t)(128 >> 4) << 32;             // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;                      // descriptor version (Blackwell)
  return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}

// x = hi + lo with hi = tf32(x), lo = tf32(x - hi): the operands of the 3xTF32 tensor-core products (hi*hi + lo*hi + hi*lo)
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  uint32_t h, l;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
  hi = __uint_as_float(h);
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(x - hi));
  lo = __uint_as_float(l);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace glamr
