// SMPL forward on sm_100a: Rodrigues + kinematic chain (pose_prep), blend shapes + pose blend + linear blend skinning
// (lbs_kernel: 1-D bulk-TMA / mbarrier double-buffered posedirs slabs, FP32 FMA, K-sparse skinning), extra joint
// regression + joint remap + re-rooting (joints_finalize).  Reference arithmetic: smplx.lbs as stated in-tree at
// HybrIK/hybrik/models/layers/smpl/lbs.py:195-288,402-548 and GLAMR's wrapper lib/models/smpl.py:289-343.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "glamr_math.cuh"
#include "smpl_model.cuh"

namespace glamr {

// ------------------------------------------------------------------------------------------------ pose_prep
// One warp per frame-person, lane j < 24 owns joint j.
//   R_j = rodrigues(pose_j)                                   lbs.py:446-477
//   J_j = j_template + j_shapedirs . beta  (== J_regressor @ v_shaped, lbs.py:240-244, by linearity)
//   G_j = G_parent(j) * [R_j | J_j - J_parent],  A_j = G_j - [0 | G_j J_j]      lbs.py:493-548
__global__ void __launch_bounds__(128) pose_prep_kernel(SmplDev m, int n, const float* __restrict__ orient,
                                                        const float* __restrict__ body_pose,
                                                        const float* __restrict__ betas, int use_betas, SmplWorkspace w) {
  const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (f >= n) return;
  pose_prep_frame(m, f, orient ? orient + (size_t)f * 3 : nullptr, body_pose + (size_t)f * 69, use_betas ? betas + (size_t)f * kNB : nullptr, w,
                  threadIdx.x & 31);
}

// ------------------------------------------------------------------------------------------------ lbs_kernel
// CTA = 128 vertices x 32 frame-persons, 128 threads (4 warps).  Warp w owns frames 8w..8w+7, lane l owns vertices
// 4l..4l+3 of the tile: a 12 (columns) x 8 (frames) register tile = 96 FP32 accumulators per thread.
//   v_posed = v_template + shapedirs.beta + posedirs^T.pose_feature           lbs.py:240,256-267
//   vert    = (sum_k w_k A_k) [v_posed; 1]                                    lbs.py:273-284
// Why this shape: the kernel is shared-memory-bandwidth bound unless the register tile is large.  Per k a thread reads
// 12 posedirs values (3 LDS.128, distinct per lane) + 8 pose-feature values (2 LDS.128, warp-broadcast) = 20 wavefronts
// per warp for 96 FFMA (0.21 wavefronts/FFMA, below the 0.25 the LSU can sustain next to 4 FFMA/clk); the first
// version (3 x 16 tile) needed 19 wavefronts per 48 FFMA and stalled on the LSU (profiles/lbs_kernel_r01.md).
// All operands arrive by 1-D bulk TMA (cp.async.bulk + mbarrier): the CTA's posedirs slab [207][384] in 23 chunks of
// 9 rows (13,824 B contiguous thanks to the tile-major re-layout), the matching [9][32] pose-feature chunk, and the
// A tile [24][32][12]; a 3-stage full/empty mbarrier ring replaces __syncthreads in the main loop.
constexpr int kFramesPerCta = 32;
constexpr int kFramesPerWarp = 8;
constexpr int kVertsPerThread = 4;
constexpr int kLbsThreads = 128;
constexpr int kMaxStages = 4;
constexpr int kChunkFloats = kChunkK * kTileCols;                 // 3456 posedirs floats per stage
constexpr uint32_t kChunkBytes = kChunkFloats * sizeof(float);    // 13,824
constexpr int kPfChunkFloats = kChunkK * kFramesPerCta;           // 288 pose-feature floats per stage
constexpr uint32_t kPfChunkBytes = kPfChunkFloats * sizeof(float);
constexpr int kATileFloats = kFramesPerCta * kNJ * 12;            // 9216
constexpr int kVpFloats = kVTile * 3 * kFramesPerCta;            // 12,288: v_posed tile handed from the GEMM phase to the skinning phase
__host__ __device__ constexpr int stage_region_floats(int stages) { return (stages * (kChunkFloats + kPfChunkFloats) > kVpFloats) ? stages * (kChunkFloats + kPfChunkFloats) : kVpFloats; }
constexpr size_t lbs_smem_bytes(int stages) { return (size_t)(stage_region_floats(stages) + kATileFloats + kFramesPerCta * kNB) * sizeof(float) + (2 * kMaxStages + 1) * sizeof(uint64_t); }

template <int KREG, int kStages>
__global__ void __launch_bounds__(kLbsThreads, 2)
lbs_kernel(SmplDev m, int n_begin, int n_end, const float* __restrict__ betas, SmplWorkspace w, float* __restrict__ vertices, int dbg) {
  constexpr int kStageRegionFloats = stage_region_floats(kStages);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* PDs = reinterpret_cast<float*>(smem_raw);              // [kStages][9][384]
  float* pfs = PDs + kStages * kChunkFloats;                     // [kStages][9][32]
  float* As = PDs + kStageRegionFloats;                          // [24][32 frames][12]
  float* bs = As + kATileFloats;                                 // [32][10]
  uint64_t* full = reinterpret_cast<uint64_t*>(bs + kFramesPerCta * kNB);   // [kStages]
  uint64_t* empty = full + kStages;                              // [kStages]
  uint64_t* abar = empty + kStages;                              // A tile

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int wf = (tid >> 5) * kFramesPerWarp;                   // first frame (within the tile) of this warp
  const int vtile = blockIdx.x;
  const int f0 = n_begin + blockIdx.y * kFramesPerCta;
  const int gv0 = vtile * kVTile + lane * kVertsPerThread;      // first of this thread's 4 vertices
  const float* pd_slab = m.pd_tiles + (size_t)vtile * kPF * kTileCols;
  const float* pf_slab = w.pf + (size_t)(f0 >> 5) * kNChunks * kPfChunkFloats;

  // issue the per-vertex constant loads first: their latency overlaps the barrier set-up and the first TMA round trip
  float sdv[kVertsPerThread][30], vt[kVertsPerThread][3];
  {
    const float4* sd4 = reinterpret_cast<const float4*>(m.shapedirs + (size_t)gv0 * 30);           // gv0 % 4 == 0 -> 480-byte aligned
    float tmp[kVertsPerThread * 30];
#pragma unroll
    for (int q = 0; q < kVertsPerThread * 30 / 4; ++q) {
      const float4 t4 = __ldg(sd4 + q);
      tmp[4 * q] = t4.x; tmp[4 * q + 1] = t4.y; tmp[4 * q + 2] = t4.z; tmp[4 * q + 3] = t4.w;
    }
#pragma unroll
    for (int v = 0; v < kVertsPerThread; ++v)
#pragma unroll
      for (int k = 0; k < 30; ++k) sdv[v][k] = tmp[v * 30 + k];
    const float4* vt4 = reinterpret_cast<const float4*>(m.v_template + (size_t)gv0 * 3);            // 12 contiguous floats
    const float4 a = __ldg(vt4), b = __ldg(vt4 + 1), c = __ldg(vt4 + 2);
    vt[0][0] = a.x; vt[0][1] = a.y; vt[0][2] = a.z; vt[1][0] = a.w; vt[1][1] = b.x; vt[1][2] = b.y;
    vt[2][0] = b.z; vt[2][1] = b.w; vt[2][2] = c.x; vt[3][0] = c.y; vt[3][1] = c.z; vt[3][2] = c.w;
  }
  float bpre[(kFramesPerCta * kNB + kLbsThreads - 1) / kLbsThreads];
#pragma unroll
  for (int i = 0; i < (kFramesPerCta * kNB + kLbsThreads - 1) / kLbsThreads; ++i) {
    const int e = tid + i * kLbsThreads;
    const int f = e / kNB, l = e - f * kNB;
    const int nn = f0 + f;
    bpre[i] = (e < kFramesPerCta * kNB && nn < n_end) ? betas[(size_t)nn * kNB + l] : 0.0f;
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kLbsThreads / 32); }
    mbar_init(abar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  auto issue_chunk = [&](int c) {      // producer: one elected thread, two bulk copies per stage
    const int s = c % kStages;
    mbar_expect_tx(&full[s], kChunkBytes + kPfChunkBytes);
    tma_bulk_g2s(PDs + s * kChunkFloats, pd_slab + (size_t)c * kChunkFloats, kChunkBytes, &full[s]);
    tma_bulk_g2s(pfs + s * kPfChunkFloats, pf_slab + (size_t)c * kPfChunkFloats, kPfChunkBytes, &full[s]);
  };
  // the first stages' posedirs slabs are requested here; their pose-feature halves and the A tile follow the shape blend below
  if (tid == 0) {
#pragma unroll
    for (int c = 0; c < kStages - 1; ++c) {
      mbar_expect_tx_only(&full[c], kChunkBytes);
      tma_bulk_g2s(PDs + c * kChunkFloats, pd_slab + (size_t)c * kChunkFloats, kChunkBytes, &full[c]);
    }
  }
#pragma unroll
  for (int i = 0; i < (kFramesPerCta * kNB + kLbsThreads - 1) / kLbsThreads; ++i) {
    const int e = tid + i * kLbsThreads;
    if (e < kFramesPerCta * kNB) bs[e] = bpre[i];
  }
  __syncthreads();

  // acc[f][c]: c = 3 * vertex + coord over the thread's 4 vertices
  float acc[kFramesPerWarp][12];
#pragma unroll
  for (int f = 0; f < kFramesPerWarp; ++f) {
    float bl[kNB];
#pragma unroll
    for (int l = 0; l < kNB; ++l) bl[l] = bs[(wf + f) * kNB + l];
#pragma unroll
    for (int v = 0; v < kVertsPerThread; ++v) {
      float a0 = vt[v][0], a1 = vt[v][1], a2 = vt[v][2];
#pragma unroll
      for (int l = 0; l < kNB; ++l) {
        a0 = fmaf(sdv[v][l], bl[l], a0);
        a1 = fmaf(sdv[v][10 + l], bl[l], a1);
        a2 = fmaf(sdv[v][20 + l], bl[l], a2);
      }
      acc[f][3 * v + 0] = a0; acc[f][3 * v + 1] = a1; acc[f][3 * v + 2] = a2;
    }
  }

  if (tid == 0) {
    mbar_expect_tx(abar, (uint32_t)kATileFloats * sizeof(float));
    tma_bulk_g2s(As, w.A + (size_t)(f0 >> 5) * kATileFloats, (uint32_t)kATileFloats * sizeof(float), abar);
#pragma unroll
    for (int c = 0; c < kStages - 1; ++c) {
      mbar_expect_tx(&full[c], kPfChunkBytes);
      tma_bulk_g2s(pfs + c * kPfChunkFloats, pf_slab + (size_t)c * kPfChunkFloats, kPfChunkBytes, &full[c]);
    }
  }

  for (int c = 0; c < kNChunks; ++c) {
    const int s = c % kStages;
    if (tid == 0 && c + kStages - 1 < kNChunks) {
      // the stage about to be refilled was last read for chunk c-1: wait until every warp released it
      if (c >= 1) mbar_wait(&empty[(c + kStages - 1) % kStages], ((c - 1) / kStages) & 1);
      issue_chunk(c + kStages - 1);
    }
    mbar_wait(&full[s], (c / kStages) & 1);
    const float4* P = reinterpret_cast<const float4*>(PDs + s * kChunkFloats + 12 * lane);
    const float4* F = reinterpret_cast<const float4*>(pfs + s * kPfChunkFloats + wf);
    if (!(GLAMR_DBG(dbg) & 1))
#pragma unroll
    for (int k = 0; k < kChunkK; ++k) {
      const float4 p0 = P[k * (kTileCols / 4) + 0], p1 = P[k * (kTileCols / 4) + 1], p2 = P[k * (kTileCols / 4) + 2];
      const float4 q0 = F[k * (kFramesPerCta / 4) + 0], q1 = F[k * (kFramesPerCta / 4) + 1];
      const float pv[12] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w, p2.x, p2.y, p2.z, p2.w};
      const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
      for (int f = 0; f < kFramesPerWarp; ++f)
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) acc[f][cc] = fmaf(qv[f], pv[cc], acc[f][cc]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }
  // ---- hand the v_posed tile to the skinning phase through shared memory (the stage buffers are free now).
  // Layout VP[row = vertex*3 + coord][32 frames] with the 4-frame chunk index XOR-swizzled by the writing lane so that
  // both the STS.128 here (lanes = vertices) and the LDS.32 below (lanes = frames) are bank-conflict free.
  __syncthreads();
  float* VP = PDs;
#pragma unroll
  for (int v = 0; v < kVertsPerThread; ++v)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      const int row = (lane * kVertsPerThread + v) * 3 + cc;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int chunk = ((wf >> 2) + h) ^ (lane & 7);
        *reinterpret_cast<float4*>(VP + row * 32 + chunk * 4) =
            make_float4(acc[4 * h + 0][3 * v + cc], acc[4 * h + 1][3 * v + cc], acc[4 * h + 2][3 * v + cc], acc[4 * h + 3][3 * v + cc]);
      }
    }
  mbar_wait(abar, 0);
  __syncthreads();

  // ---- skinning: warp w owns vertices 32w..32w+31 of the tile, lane = frame.  Joint indices / weights are
  // warp-uniform (prefetched one vertex per lane, broadcast with shuffles), a lane reads its frame's A_j with three
  // LDS.128: every LDS is conflict free.
  const int fr = lane;
  const int n = f0 + fr;
  const bool n_ok = n < n_end;
  const int vbase = (tid >> 5) * 32;
  if (!(GLAMR_DBG(dbg) & 2)) {
    if (KREG > 0) {
      const int gvl = min(vtile * kVTile + vbase + lane, kVPad - 1);
      const float4 my_w = *reinterpret_cast<const float4*>(m.skin_w + (size_t)gvl * 4);
      const unsigned int my_j = *reinterpret_cast<const unsigned int*>(m.skin_j + (size_t)gvl * 4);
      const int my_ci = m.compact_of_vertex[gvl];
#pragma unroll 4
      for (int i = 0; i < 32; ++i) {
        const int vi = vbase + i;
        const int gv = vtile * kVTile + vi;
        if (gv >= kV) break;
        const float w0 = __shfl_sync(0xffffffffu, my_w.x, i), w1 = __shfl_sync(0xffffffffu, my_w.y, i);
        const float w2 = __shfl_sync(0xffffffffu, my_w.z, i), w3 = __shfl_sync(0xffffffffu, my_w.w, i);
        const unsigned int jj = __shfl_sync(0xffffffffu, my_j, i);
        const int ci = __shfl_sync(0xffffffffu, my_ci, i);
        const int pos = ((((fr >> 2) ^ ((vi >> 2) & 7)) << 2) | (fr & 3));
        const float x = VP[(vi * 3 + 0) * 32 + pos], y = VP[(vi * 3 + 1) * 32 + pos], z = VP[(vi * 3 + 2) * 32 + pos];
        const float4* a0 = reinterpret_cast<const float4*>(As + ((jj & 0xff) * 32 + fr) * 12);
        const float4* a1 = reinterpret_cast<const float4*>(As + (((jj >> 8) & 0xff) * 32 + fr) * 12);
        const float4* a2 = reinterpret_cast<const float4*>(As + (((jj >> 16) & 0xff) * 32 + fr) * 12);
        const float4* a3 = reinterpret_cast<const float4*>(As + (((jj >> 24) & 0xff) * 32 + fr) * 12);
        float T[12];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const float4 q0 = a0[r], q1 = a1[r], q2 = a2[r], q3 = a3[r];
          T[4 * r + 0] = fmaf(w3, q3.x, fmaf(w2, q2.x, fmaf(w1, q1.x, w0 * q0.x)));
          T[4 * r + 1] = fmaf(w3, q3.y, fmaf(w2, q2.y, fmaf(w1, q1.y, w0 * q0.y)));
          T[4 * r + 2] = fmaf(w3, q3.z, fmaf(w2, q2.z, fmaf(w1, q1.z, w0 * q0.z)));
          T[4 * r + 3] = fmaf(w3, q3.w, fmaf(w2, q2.w, fmaf(w1, q1.w, w0 * q0.w)));
        }
        const float ox = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[3])));
        const float oy = fmaf(T[4], x, fmaf(T[5], y, fmaf(T[6], z, T[7])));
        const float oz = fmaf(T[8], x, fmaf(T[9], y, fmaf(T[10], z, T[11])));
        if (n_ok) {
          if (vertices) {
            float* o = vertices + ((size_t)n * kV + gv) * 3;
            o[0] = ox; o[1] = oy; o[2] = oz;
          }
          if (ci >= 0) {
            float* o = w.vcompact + ((size_t)n * m.S + ci) * 3;
            o[0] = ox; o[1] = oy; o[2] = oz;
          }
        }
      }
    } else {
      for (int vi = vbase; vi < vbase + 32; ++vi) {
        const int gv = vtile * kVTile + vi;
        if (gv >= kV) break;
        const int ci = m.compact_of_vertex[gv];
        const int pos = ((((fr >> 2) ^ ((vi >> 2) & 7)) << 2) | (fr & 3));
        const float x = VP[(vi * 3 + 0) * 32 + pos], y = VP[(vi * 3 + 1) * 32 + pos], z = VP[(vi * 3 + 2) * 32 + pos];
        float T[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) T[k] = 0.0f;
        for (int s = 0; s < m.K; ++s) {
          const int jj = m.skin_j[(size_t)gv * m.K + s];
          const float wt = m.skin_w[(size_t)gv * m.K + s];
          const float* a = As + (jj * 32 + fr) * 12;
#pragma unroll
          for (int k = 0; k < 12; ++k) T[k] = fmaf(wt, a[k], T[k]);
        }
        const float ox = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[3])));
        const float oy = fmaf(T[4], x, fmaf(T[5], y, fmaf(T[6], z, T[7])));
        const float oz = fmaf(T[8], x, fmaf(T[9], y, fmaf(T[10], z, T[11])));
        if (n_ok) {
          if (vertices) {
            float* o = vertices + ((size_t)n * kV + gv) * 3;
            o[0] = ox; o[1] = oy; o[2] = oz;
          }
          if (ci >= 0) {
            float* o = w.vcompact + ((size_t)n * m.S + ci) * 3;
            o[0] = ox; o[1] = oy; o[2] = oz;
          }
        }
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------ blend features
// The A operand of the blend GEMM for frame-person f: (R_j - I) of the 23 body joints (lbs.py:256-258), the betas, the constant 1
// that multiplies v_template and zero padding, as tf32 hi / lo in the UMMA image (see pose_prep_frame).  It depends on the body
// pose and the betas only -- NOT on the root orientation -- so the optimiser evaluates it (and the blend GEMM behind it) off the
// critical path of the iteration.  One warp per frame-person.
__global__ void __launch_bounds__(128) blend_features_kernel(int n, const float* __restrict__ body_pose, const float* __restrict__ betas, SmplWorkspace w) {
  const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (f >= n) return;
  float* tile = w.tcA + (size_t)(f >> 7) * kTcChunks * kTcAStageFloats;
  const int r = f & 127;
  auto put = [&](int k, float v) {
    float hi, lo;
    split_tf32(v, hi, lo);
    float* q = tile + (size_t)(k >> 3) * kTcAStageFloats + (((k >> 2) & 1) * kTcM + r) * 4 + (k & 3);
    q[0] = hi;
    q[kTcAStageFloats / 2] = lo;
  };
  if (lane >= 1 && lane < kNJ) {
    const float* bp = body_pose + (size_t)f * 69 + (lane - 1) * 3;
    const float rv[3] = {bp[0], bp[1], bp[2]};
    float R[9];
    rodrigues_smplx(rv, R);
#pragma unroll
    for (int k = 0; k < 9; ++k) put((lane - 1) * 9 + k, R[k] - ((k % 4 == 0) ? 1.0f : 0.0f));
  } else if (lane == 0) {
#pragma unroll
    for (int l = 0; l < kNB; ++l) put(kPF + l, betas ? betas[(size_t)f * kNB + l] : 0.0f);
    put(kPF + kNB, 1.0f);
#pragma unroll
    for (int k = kTcFeat; k < kTcK; ++k) put(k, 0.0f);
  }
}

// ------------------------------------------------------------------------------------------------ tensor-core LBS
// The shape blend + pose blend of SMPL is one contraction  v_posed[frame, col] = sum_k feat[frame, k] basis[col, k]
// (k: 207 pose features x posedirs | 10 betas x shapedirs | 1 x v_template; lbs.py:240,256-267), i.e. a [n x 218] x [218 x 20670]
// GEMM.  lbs_blend_tc_kernel runs it on the 5th-generation tensor cores with FP32 accuracy (3xTF32: hi*hi + lo*hi + hi*lo,
// |error| ~ 2e-7 on the blended vertex): both operands are PRE-SPLIT into tf32 hi / lo and pre-tiled in global memory as the UMMA
// K-major core-matrix image (basis once at glamr_smpl_create, features by pose_prep_frame), so a pipeline stage is two 1-D bulk
// TMA copies (8 KB of A, 16 KB of B) with no SIMT work on the operand path.  CTA tile = 128 frames (TMEM lanes) x 256 basis columns
// (TMEM columns), K in 28 steps of 8; warp 0 = TMA producer, warp 1 = MMA issuer (one elected thread, tcgen05.commit -> mbarrier),
// warps 2-5 = epilogue: tcgen05.ld the accumulator and store it TRANSPOSED ([column][frame]) so that lbs_skin_kernel (lanes =
// frames) reads 128 contiguous bytes per vertex coordinate.  4 stages x 24 KB = 96 KB of shared memory and 256 TMEM columns per
// CTA: two CTAs per SM overlap one's epilogue with the other's main loop.
constexpr int kTcStages = 4;
constexpr int kTcThreads = 192;
constexpr uint32_t kTcABytes = kTcAStageFloats * sizeof(float);      // 8,192
constexpr uint32_t kTcBBytes = kTcBStageFloats * sizeof(float);      // 16,384
constexpr size_t kTcSmemBytes = (size_t)kTcStages * (kTcABytes + kTcBBytes) + 128;

__global__ void __launch_bounds__(kTcThreads) lbs_blend_tc_kernel(SmplDev m, SmplWorkspace w) {
  extern __shared__ __align__(128) unsigned char tc_raw[];
  float* As = reinterpret_cast<float*>(tc_raw);                                   // [stages][hi | lo][2][128][4]
  float* Bs = As + kTcStages * kTcAStageFloats;                                   // [stages][hi | lo][2][256][4]
  uint64_t* full = reinterpret_cast<uint64_t*>(Bs + kTcStages * kTcBStageFloats); // [stages]
  uint64_t* empty = full + kTcStages;                                             // [stages]
  uint64_t* acc_full = empty + kTcStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntile = blockIdx.x, mtile = blockIdx.y;
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTcN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kTcStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(acc_full, 1);
    mbar_fence_init();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      const float* gA = w.tcA + (size_t)mtile * kTcChunks * kTcAStageFloats;
      const float* gB = m.tcB + (size_t)ntile * kTcChunks * kTcBStageFloats;
      for (int c = 0; c < kTcStages; ++c) {
        mbar_expect_tx_only(&full[c], kTcBBytes);
        tma_bulk_g2s(Bs + c * kTcBStageFloats, gB + (size_t)c * kTcBStageFloats, kTcBBytes, &full[c]);
      }
      for (int c = 0; c < kTcChunks; ++c) {
        const int s = c % kTcStages;
        if (c >= kTcStages) {
          mbar_wait(&empty[s], ((c / kTcStages) - 1) & 1);                       // the MMAs that read this stage have completed
          mbar_expect_tx(&full[s], kTcABytes + kTcBBytes);
          tma_bulk_g2s(Bs + s * kTcBStageFloats, gB + (size_t)c * kTcBStageFloats, kTcBBytes, &full[s]);
        } else {
          mbar_expect_tx(&full[s], kTcABytes);
        }
        tma_bulk_g2s(As + s * kTcAStageFloats, gA + (size_t)c * kTcAStageFloats, kTcABytes, &full[s]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2, K-major A/B, N>>3 [17,23), M>>4 [24,29)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kTcN >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);
      for (int c = 0; c < kTcChunks; ++c) {
        const int s = c % kTcStages;
        mbar_wait(&full[s], (c / kTcStages) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const float* a = As + s * kTcAStageFloats;
        const float* b = Bs + s * kTcBStageFloats;
        const uint64_t dah = umma_desc_kmajor_noswizzle(a, kTcM), dal = umma_desc_kmajor_noswizzle(a + kTcAStageFloats / 2, kTcM);
        const uint64_t dbh = umma_desc_kmajor_noswizzle(b, kTcN), dbl = umma_desc_kmajor_noswizzle(b + kTcBStageFloats / 2, kTcN);
        umma_tf32(tmem_d, dah, dbh, idesc, c > 0 ? 1u : 0u);
        umma_tf32(tmem_d, dal, dbh, idesc, 1u);
        umma_tf32(tmem_d, dah, dbl, idesc, 1u);
        // arrives on empty[s] once every MMA issued so far has completed (implies tcgen05.fence::before_thread_sync)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&empty[s])) : "memory");
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(acc_full)) : "memory");
    }
  } else {
    // ---- epilogue: warp q = warp % 4 may read TMEM lanes 32 q .. 32 q + 31 (= frames of this tile)
    mbar_wait(acc_full, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int q = warp & 3;
    const int frame = mtile * kTcM + q * 32 + lane;                              // < w.mpad by construction
    // v_posed^T [column][frame], or frame-tiled [frame / 20][column][frame % 20] for the tensor-core skinning
    float* out = w.vp_tiled ? w.vpT + ((size_t)(frame / kSkF) * kTcCols + (size_t)ntile * kTcN) * kSkF + frame % kSkF
                            : w.vpT + (size_t)ntile * kTcN * w.mpad + frame;
    const size_t cstride = w.vp_tiled ? (size_t)kSkF : (size_t)w.mpad;
#pragma unroll 1
    for (int cc = 0; cc < kTcN / 32; ++cc) {
      uint32_t v[32];
      const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(cc * 32);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, "
          "%28, %29, %30, %31}, [%32];\n"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
            "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
            "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
            "=r"(v[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 32; ++j) out[(size_t)(cc * 32 + j) * cstride] = __uint_as_float(v[j]);   // 32 lanes = 32 consecutive frames: 128 B per column (2-3 runs when tiled)
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(kTcN));
}

// Skinning of the blended vertices (lbs.py:273-284): CTA = 128 vertices x 32 frames, warp = 32 vertices, lane = frame.
// The tile's relative joint transforms [24][32][12] arrive by one bulk TMA copy; joint indices / weights are warp-uniform
// (prefetched one vertex per lane, broadcast by shuffles); v_posed comes from the transposed blend output with one coalesced
// 128-byte load per vertex coordinate; a lane reads its frame's A_j with three conflict-free LDS.128.
constexpr size_t kSkinSmemBytes = (size_t)kATileFloats * sizeof(float) + 16;
template <int KREG>
__global__ void __launch_bounds__(kLbsThreads) lbs_skin_kernel(SmplDev m, int n_begin, int n_end, SmplWorkspace w, float* __restrict__ vertices) {
  extern __shared__ __align__(128) unsigned char skin_raw[];
  float* As = reinterpret_cast<float*>(skin_raw);
  uint64_t* abar = reinterpret_cast<uint64_t*>(As + kATileFloats);
  const int tid = threadIdx.x, lane = tid & 31;
  const int vtile = blockIdx.x;
  const int f0 = n_begin + blockIdx.y * kFramesPerCta;
  if (tid == 0) {
    mbar_init(abar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  const int vbase = (tid >> 5) * 32;
  const int gvl = min(vtile * kVTile + vbase + lane, kVPad - 1);
  float4 my_w = make_float4(0.f, 0.f, 0.f, 0.f);
  unsigned int my_j = 0;
  if (KREG > 0) {
    my_w = *reinterpret_cast<const float4*>(m.skin_w + (size_t)gvl * 4);
    my_j = *reinterpret_cast<const unsigned int*>(m.skin_j + (size_t)gvl * 4);
  }
  const int my_ci = m.compact_of_vertex[gvl];
  if (tid == 0) {
    mbar_expect_tx(abar, (uint32_t)kATileFloats * sizeof(float));
    tma_bulk_g2s(As, w.A + (size_t)(f0 >> 5) * kATileFloats, (uint32_t)kATileFloats * sizeof(float), abar);
  }
  const int fr = lane;
  const int n = f0 + fr;
  const bool n_ok = n < n_end;
  mbar_wait(abar, 0);
  const float* vp = w.vpT + (size_t)(vtile * kVTile + vbase) * 3 * w.mpad + n;      // n < mpad (frames padded to 128)
  constexpr int U = 4;
#pragma unroll 1
  for (int i0 = 0; i0 < 32; i0 += U) {
    float x[U], y[U], z[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int gv = vtile * kVTile + vbase + i0 + u;
      const bool ok = gv < kV;
      const float* q = vp + (size_t)(i0 + u) * 3 * w.mpad;
      x[u] = ok ? q[0] : 0.0f;
      y[u] = ok ? q[w.mpad] : 0.0f;
      z[u] = ok ? q[2 * (size_t)w.mpad] : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u;
      const int gv = vtile * kVTile + vbase + i;
      if (gv >= kV) break;
      const int ci = __shfl_sync(0xffffffffu, my_ci, i);
      float T[12];
      if (KREG > 0) {
        const float w0 = __shfl_sync(0xffffffffu, my_w.x, i), w1 = __shfl_sync(0xffffffffu, my_w.y, i);
        const float w2 = __shfl_sync(0xffffffffu, my_w.z, i), w3 = __shfl_sync(0xffffffffu, my_w.w, i);
        const unsigned int jj = __shfl_sync(0xffffffffu, my_j, i);
        const float4* a0 = reinterpret_cast<const float4*>(As + ((jj & 0xff) * 32 + fr) * 12);
        const float4* a1 = reinterpret_cast<const float4*>(As + (((jj >> 8) & 0xff) * 32 + fr) * 12);
        const float4* a2 = reinterpret_cast<const float4*>(As + (((jj >> 16) & 0xff) * 32 + fr) * 12);
        const float4* a3 = reinterpret_cast<const float4*>(As + (((jj >> 24) & 0xff) * 32 + fr) * 12);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const float4 q0 = a0[r], q1 = a1[r], q2 = a2[r], q3 = a3[r];
          T[4 * r + 0] = fmaf(w3, q3.x, fmaf(w2, q2.x, fmaf(w1, q1.x, w0 * q0.x)));
          T[4 * r + 1] = fmaf(w3, q3.y, fmaf(w2, q2.y, fmaf(w1, q1.y, w0 * q0.y)));
          T[4 * r + 2] = fmaf(w3, q3.z, fmaf(w2, q2.z, fmaf(w1, q1.z, w0 * q0.z)));
          T[4 * r + 3] = fmaf(w3, q3.w, fmaf(w2, q2.w, fmaf(w1, q1.w, w0 * q0.w)));
        }
      } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) T[k] = 0.0f;
        for (int sidx = 0; sidx < m.K; ++sidx) {
          const int jj = m.skin_j[(size_t)gv * m.K + sidx];
          const float wt = m.skin_w[(size_t)gv * m.K + sidx];
          const float* a = As + (jj * 32 + fr) * 12;
#pragma unroll
          for (int k = 0; k < 12; ++k) T[k] = fmaf(wt, a[k], T[k]);
        }
      }
      const float ox = fmaf(T[0], x[u], fmaf(T[1], y[u], fmaf(T[2], z[u], T[3])));
      const float oy = fmaf(T[4], x[u], fmaf(T[5], y[u], fmaf(T[6], z[u], T[7])));
      const float oz = fmaf(T[8], x[u], fmaf(T[9], y[u], fmaf(T[10], z[u], T[11])));
      if (n_ok) {
        if (vertices) {
          float* o = vertices + ((size_t)n * kV + gv) * 3;
          o[0] = ox; o[1] = oy; o[2] = oz;
        }
        if (ci >= 0) {
          float* o = w.vcompact + ((size_t)n * m.S + ci) * 3;
          o[0] = ox; o[1] = oy; o[2] = oz;
        }
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------ tensor-core skinning
// lbs.py:273-284 as a GEMM with a fused epilogue.  The blended transform of vertex v in frame f is T[v][f] = sum_j W[v][j] A_j[f]
// (12 numbers), i.e. [128 vertices x 24 joints] x [24 joints x (20 frames x 12)] per CTA: M = 128 (TMEM lanes = vertices), N = 240
// (TMEM columns), K = 24 in three kind::tf32 steps, 3xTF32 (hi*hi + lo*hi + hi*lo) like the blend.  Both operands are pre-tiled
// UMMA images (W: model constant built at glamr_smpl_create; A: written by pose_prep_frame), so the whole operand traffic of a
// CTA is three bulk copies: W image 24 KB, A image 45 KB, and the 128 x 20 v_posed block 30 KB (the blend stores v_posed frame-
// tiled for this).  Epilogue: thread = vertex reads its 12 x 20 transform entries with tcgen05.ld, its v_posed with conflict-free
// LDS.128 (80-byte row pitch, 240-byte lane stride) and applies T to it -- no shared-memory traffic for the joint transforms,
// which bounded the SIMT skinning (12 LDS.128 per vertex-frame).  warp 0 = producer, warp 1 = TMEM + MMA, warps 2-5 = epilogue;
// 101 KB of shared memory and 256 TMEM columns per CTA: two CTAs per SM overlap one's epilogue with the other's loads.
constexpr uint32_t kSkWBytes = kSkWImageFloats * sizeof(float);       // 24,576
constexpr uint32_t kSkBBytes = kSkBImageFloats * sizeof(float);       // 46,080
constexpr uint32_t kSkVBytes = kSkVpTileFloats * sizeof(float);       // 30,720
constexpr size_t kSkinTcSmemBytes = (size_t)kSkWBytes + kSkBBytes + kSkVBytes + 128;

#define GLAMR_TMEM_LD_X16(v, taddr)                                                                                                  \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n" \
               : "=r"((v)[0]), "=r"((v)[1]), "=r"((v)[2]), "=r"((v)[3]), "=r"((v)[4]), "=r"((v)[5]), "=r"((v)[6]), "=r"((v)[7]),      \
                 "=r"((v)[8]), "=r"((v)[9]), "=r"((v)[10]), "=r"((v)[11]), "=r"((v)[12]), "=r"((v)[13]), "=r"((v)[14]), "=r"((v)[15])  \
               : "r"(taddr))

#define GLAMR_TMEM_LD_X8(v, taddr)                                                                                  \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"                      \
               : "=r"((v)[0]), "=r"((v)[1]), "=r"((v)[2]), "=r"((v)[3]), "=r"((v)[4]), "=r"((v)[5]), "=r"((v)[6]), "=r"((v)[7]) \
               : "r"(taddr))

constexpr int kSkinTcThreads = 320;     // warp 0 producer, warp 1 TMEM + MMA, warps 2-9 epilogue (two warps per TMEM lane quarter)
constexpr int kSkTilesPerCta = 3;       // frame tiles one CTA sweeps (W stays in shared memory; 54 x 5 CTAs = one wave at 300 frames)

__global__ void __launch_bounds__(kSkinTcThreads) lbs_skin_tc_kernel(SmplDev m, int n, SmplWorkspace w, float* __restrict__ vertices) {
  extern __shared__ __align__(128) unsigned char sk_raw[];
  float* Ws = reinterpret_cast<float*>(sk_raw);                       // [hi | lo][6][128][4]
  float* Bs = Ws + kSkWImageFloats;                                   // [hi | lo][6][240][4]
  float* Vs = Bs + kSkBImageFloats;                                   // [384 rows = vertex * 3 + coordinate][20 frames]
  uint64_t* full_w = reinterpret_cast<uint64_t*>(Vs + kSkVpTileFloats);
  uint64_t* full_b = full_w + 1;          // A image of the current frame tile has landed
  uint64_t* full_v = full_w + 2;          // v_posed block has landed
  uint64_t* acc_full = full_w + 3;        // the tile's MMAs have completed (accumulator readable)
  uint64_t* b_empty = full_w + 4;         // ... and no longer read Bs: the next A image may be fetched
  uint64_t* v_empty = full_w + 5;         // the 4 epilogue warps are done with Vs
  uint64_t* acc_empty = full_w + 6;       // ... and with the accumulator
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full_w + 7);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int vtile = blockIdx.x;
  const int ftile0 = blockIdx.y * kSkTilesPerCta;
  const int ntiles = min(kSkTilesPerCta, (n + kSkF - 1) / kSkF - ftile0);
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  if (tid == 0) {
    mbar_init(full_w, 1);
    mbar_init(full_b, 1);
    mbar_init(full_v, 1);
    mbar_init(acc_full, 1);
    mbar_init(b_empty, 1);
    mbar_init(v_empty, 8);
    mbar_init(acc_empty, 8);
    mbar_fence_init();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(full_w, kSkWBytes);
      tma_bulk_g2s(Ws, m.skW + (size_t)vtile * kSkWImageFloats, kSkWBytes, full_w);
      for (int it = 0; it < ntiles; ++it) {
        const int ftile = ftile0 + it;
        if (it > 0) mbar_wait(b_empty, (it - 1) & 1);
        mbar_expect_tx(full_b, kSkBBytes);
        tma_bulk_g2s(Bs, w.skB + (size_t)ftile * kSkBImageFloats, kSkBBytes, full_b);
        if (it > 0) mbar_wait(v_empty, (it - 1) & 1);
        mbar_expect_tx(full_v, kSkVBytes);
        tma_bulk_g2s(Vs, w.vpT + ((size_t)ftile * kTcCols + (size_t)vtile * kTileCols) * kSkF, kSkVBytes, full_v);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kSkN >> 3) << 17) | ((uint32_t)(kVTile >> 4) << 24);
      mbar_wait(full_w, 0);
      for (int it = 0; it < ntiles; ++it) {
        mbar_wait(full_b, it & 1);
        if (it > 0) mbar_wait(acc_empty, (it - 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int c = 0; c < kNJ / 8; ++c) {
          const float* a = Ws + c * 2 * kVTile * 4;
          const float* b = Bs + c * 2 * kSkN * 4;
          const uint64_t dah = umma_desc_kmajor_noswizzle(a, kVTile), dal = umma_desc_kmajor_noswizzle(a + kSkWHalf, kVTile);
          const uint64_t dbh = umma_desc_kmajor_noswizzle(b, kSkN), dbl = umma_desc_kmajor_noswizzle(b + kSkBHalf, kSkN);
          umma_tf32(tmem_d, dah, dbh, idesc, c > 0 ? 1u : 0u);
          umma_tf32(tmem_d, dal, dbh, idesc, 1u);
          umma_tf32(tmem_d, dah, dbl, idesc, 1u);
        }
        // both arrive once every MMA issued so far has completed
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(b_empty)) : "memory");
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(acc_full)) : "memory");
      }
    }
  } else {
    // ---- epilogue: warp q = warp % 4 may read TMEM lanes 32 q .. 32 q + 31 (= vertices of this tile); the two warps of a quarter take
    // alternate pairs of frames (24 accumulator columns each)
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int vl = q * 32 + lane;
    const int gv = vtile * kVTile + vl;
    const bool v_ok = gv < kV;
    const int ci = m.compact_of_vertex[min(gv, kVPad - 1)];
    const float* vrow = Vs + (size_t)vl * 3 * kSkF;
    for (int it = 0; it < ntiles; ++it) {
      const int ftile = ftile0 + it;
      mbar_wait(full_v, it & 1);
      mbar_wait(acc_full, it & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
      for (int g = half; g < kSkF / 2; g += 2) {                   // 2 frames = 24 accumulator columns per step
        uint32_t t[24];
        const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * 24);
        GLAMR_TMEM_LD_X16(t, taddr);
        GLAMR_TMEM_LD_X8(t + 16, taddr + 16);
        const float2 xs = *reinterpret_cast<const float2*>(vrow + g * 2);
        const float2 ys = *reinterpret_cast<const float2*>(vrow + kSkF + g * 2);
        const float2 zs = *reinterpret_cast<const float2*>(vrow + 2 * kSkF + g * 2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const float x[2] = {xs.x, xs.y}, y[2] = {ys.x, ys.y}, z[2] = {zs.x, zs.y};
#pragma unroll
        for (int ff = 0; ff < 2; ++ff) {
          const int fl = ftile * kSkF + g * 2 + ff;                // local frame-person index
#define GLAMR_T(k) __uint_as_float(t[ff * 12 + (k)])
          const float ox = fmaf(GLAMR_T(0), x[ff], fmaf(GLAMR_T(1), y[ff], fmaf(GLAMR_T(2), z[ff], GLAMR_T(3))));
          const float oy = fmaf(GLAMR_T(4), x[ff], fmaf(GLAMR_T(5), y[ff], fmaf(GLAMR_T(6), z[ff], GLAMR_T(7))));
          const float oz = fmaf(GLAMR_T(8), x[ff], fmaf(GLAMR_T(9), y[ff], fmaf(GLAMR_T(10), z[ff], GLAMR_T(11))));
#undef GLAMR_T
          if (fl < n && v_ok) {
            if (vertices) {
              float* o = vertices + ((size_t)fl * kV + gv) * 3;
              o[0] = ox; o[1] = oy; o[2] = oz;
            }
            if (ci >= 0) {
              float* o = w.vcompact + ((size_t)fl * m.S + ci) * 3;
              o[0] = ox; o[1] = oy; o[2] = oz;
            }
          }
        }
      }
      // release the accumulator and the v_posed block for the next frame tile
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(acc_empty);
        mbar_arrive(v_empty);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(256));
}

// ------------------------------------------------------------------------------------------------ joints_finalize
// One warp per frame-person: gather the mapped joints from [24 LBS | picks | extra regressed], re-root at joint 0
// and apply scale / root translation   (lib/models/smpl.py:299-315)
__global__ void __launch_bounds__(128) joints_finalize_kernel(SmplDev m, int n, int orig_joints, const float* __restrict__ root_trans,
                                                              const float* __restrict__ root_scale, SmplWorkspace w,
                                                              float* __restrict__ joints) {
  const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (f >= n) return;
  const int n_out = orig_joints ? kNJ : m.n_map;
  float root[3];
  raw_joint(m, w, f, orig_joints ? 0 : m.joint_map[0], root);
  if (lane == 0) {
    w.root_raw[f * 3 + 0] = root[0]; w.root_raw[f * 3 + 1] = root[1]; w.root_raw[f * 3 + 2] = root[2];
  }
  const float sc = (root_trans && root_scale) ? root_scale[f] : 1.0f;
  for (int k = lane; k < n_out; k += 32) {
    float v[3];
    raw_joint(m, w, f, orig_joints ? k : m.joint_map[k], v);
    float* o = joints + ((size_t)f * n_out + k) * 3;
    if (root_trans) {
      o[0] = (v[0] - root[0]) * sc + root_trans[f * 3 + 0];
      o[1] = (v[1] - root[1]) * sc + root_trans[f * 3 + 1];
      o[2] = (v[2] - root[2]) * sc + root_trans[f * 3 + 2];
    } else {
      o[0] = v[0]; o[1] = v[1]; o[2] = v[2];
    }
  }
}

__global__ void reroot_vertices_kernel(int n, const float* __restrict__ root_raw, const float* __restrict__ root_trans,
                                       const float* __restrict__ root_scale, float* __restrict__ vertices) {
  const size_t total = (size_t)n * kV * 3;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int f = (int)(e / (kV * 3));
    const int c = (int)(e % 3);
    const float sc = root_scale ? root_scale[f] : 1.0f;
    vertices[e] = (vertices[e] - root_raw[f * 3 + c]) * sc + root_trans[f * 3 + c];
  }
}

// fk-only joints (SMPL.get_joints): re-root the posed LBS joints
__global__ void fk24_finalize_kernel(int n, const float* __restrict__ jposed, const float* __restrict__ root_trans,
                                     const float* __restrict__ root_scale, float* __restrict__ joints) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * kNJ * 3) return;
  const int f = e / (kNJ * 3), c = e % 3;
  float v = jposed[e];
  if (root_trans) {
    const float sc = root_scale ? root_scale[f] : 1.0f;
    v = (v - jposed[(size_t)f * kNJ * 3 + c]) * sc + root_trans[f * 3 + c];
  }
  joints[e] = v;
}

// ------------------------------------------------------------------------------------------------ launches
int launch_pose_prep(const SmplDev& m, int n, const float* orient, const float* body_pose, const float* betas, int use_betas,
                     const SmplWorkspace& w, cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  pose_prep_kernel<<<(n + 3) / 4, 128, 0, s>>>(m, n, orient, body_pose, betas, use_betas, w);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

// An SM runs with ONE L1 / shared-memory split at a time.  blend_features_kernel / pose_prep_kernel have no dynamic shared memory, so by
// default they run with a small shared-memory split, and the GEMM kernel that follows each of them in its stream (2 x 96-101 KB per SM)
// can only be placed on an SM after the small kernel's CTAs have drained and the SM has been re-configured.  Asking for the maximal
// shared-memory split on the small SMPL kernels too removes that hand-over: 193.0 -> 157.4 us per iteration at 4 x 300 frame-persons
// (no change at 1 x 300).  The optimiser's own small kernels lose more from the smaller L1 than they gain (+6 us at 1 x 300), so they
// keep the default split.
static int lbs_set_attrs() {
  static bool attrs = false;
  if (!attrs) {
    attrs = true;
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_blend_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_skin_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(blend_features_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(pose_prep_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_blend_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_skin_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSkinSmemBytes));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_skin_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSkinSmemBytes));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_skin_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSkinTcSmemBytes));
  }
  return GLAMR_OK;
}
// the A operand of the blend GEMM for local frame-persons [0, n)
int launch_blend_features(int n, const float* body_pose, const float* betas, const SmplWorkspace& w, cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  int rc;
  if ((rc = lbs_set_attrs())) return rc;
  blend_features_kernel<<<(n + 3) / 4, 128, 0, s>>>(n, body_pose, betas, w);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}
// blend GEMM for local frame-persons [0, n) from the workspace's features: v_posed (transposed) of the workspace
int launch_blend_gemm(const SmplDev& m, int n, const SmplWorkspace& w, cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  int rc;
  if ((rc = lbs_set_attrs())) return rc;
  lbs_blend_tc_kernel<<<dim3(kTcNTiles, (n + kTcM - 1) / kTcM), kTcThreads, kTcSmemBytes, s>>>(m, w);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}
int launch_blend(const SmplDev& m, int n, const float* body_pose, const float* betas, const SmplWorkspace& w, cudaStream_t s) {
  int rc;
  if ((rc = launch_blend_features(n, body_pose, betas, w, s))) return rc;
  return launch_blend_gemm(m, n, w, s);
}
// skinning of local frame-persons [0, n) from the workspace's v_posed and A
int launch_skin(const SmplDev& m, int n, const SmplWorkspace& w, float* vertices, cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  int rc;
  if ((rc = lbs_set_attrs())) return rc;
  if (w.vp_tiled) {
    lbs_skin_tc_kernel<<<dim3(kNVTiles, ((n + kSkF - 1) / kSkF + kSkTilesPerCta - 1) / kSkTilesPerCta), kSkinTcThreads, kSkinTcSmemBytes, s>>>(m, n, w, vertices);
    GLAMR_LAUNCH_CHECK();
    return GLAMR_OK;
  }
  dim3 grid(kNVTiles, (n + kFramesPerCta - 1) / kFramesPerCta);
  if (m.K == 4) lbs_skin_kernel<4><<<grid, kLbsThreads, kSkinSmemBytes, s>>>(m, 0, n, w, vertices);
  else lbs_skin_kernel<0><<<grid, kLbsThreads, kSkinSmemBytes, s>>>(m, 0, n, w, vertices);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

static int g_lbs_path = -1;
int lbs_path() {
  if (g_lbs_path < 0) {
    const char* e = getenv("GLAMR_LBS_PATH");
    g_lbs_path = e ? (strcmp(e, "tc") == 0 ? 2 : strcmp(e, "tcblend") == 0 ? 1 : 0) : GLAMR_DEFAULT_LBS_TC;
  }
  return g_lbs_path;
}
int lbs_kernel_count(const SmplDev& m) { return (lbs_path() >= 1 && m.tcB) ? 2 : 1; }

int launch_lbs(const SmplDev& m, int n_begin, int n_end, const float* betas, const SmplWorkspace& w, float* vertices, cudaStream_t s) {
  if (n_end <= n_begin) return GLAMR_OK;
  if (n_begin % kFramesPerCta != 0) return GLAMR_EINVAL;   // the tile-major scratch is indexed by whole frame tiles
  dim3 grid(kNVTiles, (n_end - n_begin + kFramesPerCta - 1) / kFramesPerCta);
  const int path = lbs_path();             // >= 1: tensor-core blend GEMM + skinning kernel (2: tensor-core skinning), 0: the one-kernel FP32 SIMT path
  {
    const int rc = lbs_set_attrs();
    if (rc) return rc;
  }
  if (path >= 1 && m.tcB && w.tcA && n_begin == 0) {
    const int mtiles = (n_end + kTcM - 1) / kTcM;
    lbs_blend_tc_kernel<<<dim3(kTcNTiles, mtiles), kTcThreads, kTcSmemBytes, s>>>(m, w);
    GLAMR_LAUNCH_CHECK();
    if (w.vp_tiled) {
      const dim3 sgrid(kNVTiles, ((n_end + kSkF - 1) / kSkF + kSkTilesPerCta - 1) / kSkTilesPerCta);
      lbs_skin_tc_kernel<<<sgrid, kSkinTcThreads, kSkinTcSmemBytes, s>>>(m, n_end, w, vertices);
    } else if (m.K == 4) {
      lbs_skin_kernel<4><<<grid, kLbsThreads, kSkinSmemBytes, s>>>(m, n_begin, n_end, w, vertices);
    } else {
      lbs_skin_kernel<0><<<grid, kLbsThreads, kSkinSmemBytes, s>>>(m, n_begin, n_end, w, vertices);
    }
    GLAMR_LAUNCH_CHECK();
    return GLAMR_OK;
  }
  static bool attrs = false;
  static int dbg = 0;
  if (!attrs) {
    attrs = true;
#ifdef GLAMR_EXPERIMENT
    const char* d = getenv("GLAMR_LBS_DEBUG");      // experiment build only: bit0 skips the FMA loop, bit1 the skinning phase
    dbg = d ? atoi(d) : 0;
#endif
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_kernel<4, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lbs_smem_bytes(3)));
    GLAMR_CUDA_TRY(cudaFuncSetAttribute(lbs_kernel<0, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lbs_smem_bytes(3)));
  }
  if (m.K == 4) lbs_kernel<4, 3><<<grid, kLbsThreads, lbs_smem_bytes(3), s>>>(m, n_begin, n_end, betas, w, vertices, dbg);
  else lbs_kernel<0, 3><<<grid, kLbsThreads, lbs_smem_bytes(3), s>>>(m, n_begin, n_end, betas, w, vertices, dbg);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

int launch_joints_finalize(const SmplDev& m, int n, int orig_joints, const float* root_trans, const float* root_scale,
                           const SmplWorkspace& w, float* joints, cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  joints_finalize_kernel<<<(n + 3) / 4, 128, 0, s>>>(m, n, orig_joints, root_trans, root_scale, w, joints);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

int launch_reroot_vertices(int n, const float* root_raw, const float* root_trans, const float* root_scale, float* vertices,
                           cudaStream_t s) {
  if (n <= 0) return GLAMR_OK;
  const size_t total = (size_t)n * kV * 3;
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  reroot_vertices_kernel<<<blocks, 256, 0, s>>>(n, root_raw, root_trans, root_scale, vertices);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

}  // namespace glamr

// =================================================================================================== C ABI
using namespace glamr;

namespace {
template <typename T>
int upload(glamr_smpl* h, const std::vector<T>& host, const T** dev) {
  void* p = nullptr;
  GLAMR_CUDA_TRY(cudaMalloc(&p, host.size() * sizeof(T) + 256));
  GLAMR_CUDA_TRY(cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
  h->allocs[h->n_allocs++] = p;
  *dev = (const T*)p;
  return GLAMR_OK;
}
}  // namespace

extern "C" int glamr_version(void) { return 100; }

extern "C" int glamr_device_sm_count(void) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  return sms;
}

extern "C" int glamr_smpl_create(glamr_smpl_t** out, const float* v_template, const float* shapedirs, const float* posedirs,
                                 const float* J_regressor, const float* lbs_weights, const int32_t* parents,
                                 const float* J_regressor_extra, int n_extra, const int32_t* pick_vertex_ids, int n_picks,
                                 const int32_t* joint_map, int n_map) {
  if (!out || !v_template || !shapedirs || !posedirs || !J_regressor || !lbs_weights || !parents || !joint_map) return GLAMR_EINVAL;
  if (n_extra < 0 || n_picks < 0 || n_map <= 0 || (n_extra > 0 && !J_regressor_extra) || (n_picks > 0 && !pick_vertex_ids)) return GLAMR_EINVAL;
  for (int k = 0; k < n_map; ++k)
    if (joint_map[k] < 0 || joint_map[k] >= kNJ + n_picks + n_extra) return GLAMR_EINVAL;
  for (int k = 0; k < n_picks; ++k)
    if (pick_vertex_ids[k] < 0 || pick_vertex_ids[k] >= kV) return GLAMR_EINVAL;
  glamr_smpl* h = (glamr_smpl*)calloc(1, sizeof(glamr_smpl));
  if (!h) return GLAMR_EINVAL;
  SmplDev& d = h->dev;
  // kinematic tree levels
  for (int j = 0; j < kNJ; ++j) d.parents[j] = parents[j];
  d.n_levels = 0;
  for (int j = 0; j < kNJ; ++j) {
    if (j > 0 && (parents[j] < 0 || parents[j] >= j)) { free(h); return GLAMR_EINVAL; }
    d.level[j] = (j == 0) ? 0 : d.level[parents[j]] + 1;
    if (d.level[j] + 1 > d.n_levels) d.n_levels = d.level[j] + 1;
  }
  d.n_extra = n_extra; d.n_picks = n_picks; d.n_map = n_map;
  int rc = GLAMR_OK;
  {  // posedirs -> [tile][k][384]
    std::vector<float> t((size_t)kNVTiles * kPF * kTileCols, 0.0f);
    for (int tile = 0; tile < kNVTiles; ++tile)
      for (int k = 0; k < kPF; ++k) {
        const int c0 = tile * kTileCols;
        const int ncol = (c0 + kTileCols <= kV * 3) ? kTileCols : (kV * 3 - c0);
        memcpy(&t[((size_t)tile * kPF + k) * kTileCols], posedirs + (size_t)k * kV * 3 + c0, ncol * sizeof(float));
      }
    if ((rc = upload(h, t, &d.pd_tiles))) goto fail;
  }
  {  // blend basis [20736 cols][224 k] = posedirs^T | shapedirs | v_template, tf32 hi / lo, UMMA K-major core-matrix image per
     // (256-column tile, 8-wide K chunk): [hi | lo][k group (4 wide)][256 cols][4]
    auto tf32_rna = [](float x) {            // cvt.rna.tf32.f32: round to nearest, ties away from zero, 10-bit mantissa
      uint32_t u;
      memcpy(&u, &x, 4);
      u = (u + 0x1000u) & 0xFFFFE000u;
      float r;
      memcpy(&r, &u, 4);
      return r;
    };
    std::vector<float> img((size_t)kTcNTiles * kTcChunks * kTcBStageFloats, 0.0f);
    for (int col = 0; col < kV * 3; ++col) {
      const int tile = col / kTcN, r = col % kTcN;
      for (int k = 0; k < kTcFeat; ++k) {
        float v;
        if (k < kPF) v = posedirs[(size_t)k * kV * 3 + col];
        else if (k < kPF + kNB) v = shapedirs[(size_t)col * kNB + (k - kPF)];      // shapedirs [v][c][l] = [col][l]
        else v = v_template[col];
        const float hi = tf32_rna(v), lo = tf32_rna(v - hi);
        float* q = &img[((size_t)tile * kTcChunks + (k >> 3)) * kTcBStageFloats + ((((k >> 2) & 1) * kTcN + r) * 4) + (k & 3)];
        q[0] = hi;
        q[kTcBStageFloats / 2] = lo;
      }
    }
    if ((rc = upload(h, img, &d.tcB))) goto fail;
    // dense skinning weights W[v][24] as the A operand of the tensor-core skinning: per 128-vertex tile [hi | lo][joint group][vertex][4]
    std::vector<float> wimg((size_t)kNVTiles * kSkWImageFloats, 0.0f);
    for (int v = 0; v < kV; ++v)
      for (int j = 0; j < kNJ; ++j) {
        const float x = lbs_weights[(size_t)v * kNJ + j];
        const float hi = tf32_rna(x), lo = tf32_rna(x - hi);
        float* q = &wimg[(size_t)(v / kVTile) * kSkWImageFloats + ((size_t)(j >> 2) * kVTile + v % kVTile) * 4 + (j & 3)];
        q[0] = hi;
        q[kSkWHalf] = lo;
      }
    if ((rc = upload(h, wimg, &d.skW))) goto fail;
  }
  {
    std::vector<float> vt((size_t)kVPad * 3, 0.0f), sd((size_t)kVPad * 30, 0.0f);
    memcpy(vt.data(), v_template, (size_t)kV * 3 * sizeof(float));
    memcpy(sd.data(), shapedirs, (size_t)kV * 30 * sizeof(float));
    if ((rc = upload(h, vt, &d.v_template))) goto fail;
    if ((rc = upload(h, sd, &d.shapedirs))) goto fail;
  }
  {  // rest joints as an affine function of beta (double accumulation on the host)
    std::vector<float> jt(kNJ * 3), js(kNJ * 3 * kNB);
    for (int j = 0; j < kNJ; ++j)
      for (int c = 0; c < 3; ++c) {
        double a = 0.0;
        double b[kNB] = {0};
        for (int v = 0; v < kV; ++v) {
          const double wv = J_regressor[(size_t)j * kV + v];
          if (wv == 0.0) continue;
          a += wv * v_template[v * 3 + c];
          for (int l = 0; l < kNB; ++l) b[l] += wv * shapedirs[((size_t)v * 3 + c) * kNB + l];
        }
        jt[j * 3 + c] = (float)a;
        for (int l = 0; l < kNB; ++l) js[(j * 3 + c) * kNB + l] = (float)b[l];
      }
    if ((rc = upload(h, jt, &d.j_template))) goto fail;
    if ((rc = upload(h, js, &d.j_shapedirs))) goto fail;
  }
  {  // K-sparse skinning weights
    int K = 1;
    for (int v = 0; v < kV; ++v) {
      int c = 0;
      for (int j = 0; j < kNJ; ++j) c += lbs_weights[(size_t)v * kNJ + j] != 0.0f;
      if (c > K) K = c;
    }
    if (K < 4) K = 4;
    d.K = K;
    std::vector<float> sw((size_t)kVPad * K, 0.0f);
    std::vector<uint8_t> sj((size_t)kVPad * K, 0);
    for (int v = 0; v < kV; ++v) {
      int c = 0;
      for (int j = 0; j < kNJ; ++j) {
        const float wv = lbs_weights[(size_t)v * kNJ + j];
        if (wv != 0.0f) { sw[(size_t)v * K + c] = wv; sj[(size_t)v * K + c] = (uint8_t)j; ++c; }
      }
    }
    if ((rc = upload(h, sw, &d.skin_w))) goto fail;
    if ((rc = upload(h, sj, &d.skin_j))) goto fail;
  }
  {  // support list + CSR of the extra regressor
    std::vector<int32_t> cov(kVPad, -1), sup;
    auto touch = [&](int v) { if (cov[v] < 0) { cov[v] = (int32_t)sup.size(); sup.push_back(v); } };
    for (int k = 0; k < n_picks; ++k) touch(pick_vertex_ids[k]);
    std::vector<int32_t> ptr(n_extra + 1, 0), ci;
    std::vector<float> rw;
    for (int r = 0; r < n_extra; ++r) {
      for (int v = 0; v < kV; ++v) {
        const float wv = J_regressor_extra[(size_t)r * kV + v];
        if (wv != 0.0f) { touch(v); ci.push_back(cov[v]); rw.push_back(wv); }
      }
      ptr[r + 1] = (int32_t)ci.size();
    }
    if (ci.empty()) { ci.push_back(0); rw.push_back(0.0f); }
    if (sup.empty()) touch(0);
    d.S = (int)sup.size();
    std::vector<int32_t> pci(n_picks > 0 ? n_picks : 1, 0), jm(joint_map, joint_map + n_map);
    for (int k = 0; k < n_picks; ++k) pci[k] = cov[pick_vertex_ids[k]];
    if ((rc = upload(h, cov, &d.compact_of_vertex))) goto fail;
    if ((rc = upload(h, ptr, &d.reg_ptr))) goto fail;
    if ((rc = upload(h, ci, &d.reg_ci))) goto fail;
    if ((rc = upload(h, rw, &d.reg_w))) goto fail;
    if ((rc = upload(h, pci, &d.pick_ci))) goto fail;
    if ((rc = upload(h, jm, &d.joint_map))) goto fail;
  }
  *out = h;
  return GLAMR_OK;
fail:
  glamr_smpl_destroy(h);
  return rc;
}

extern "C" int glamr_smpl_destroy(glamr_smpl_t* m) {
  if (!m) return GLAMR_OK;
  for (int i = 0; i < m->n_allocs; ++i) cudaFree(m->allocs[i]);
  free(m);
  return GLAMR_OK;
}

extern "C" int glamr_smpl_set_lbs_path(int path) {
  if (path < -1 || path > 2) return GLAMR_EINVAL;     // -1: back to the default (GLAMR_LBS_PATH or the compile-time choice)
  g_lbs_path = path;
  return GLAMR_OK;
}

extern "C" int glamr_smpl_info(const glamr_smpl_t* m, int what) {
  if (!m) return GLAMR_EINVAL;
  switch (what) {
    case 0: return m->dev.K;
    case 1: return m->dev.S;
    case 2: return m->dev.n_map;
    default: return GLAMR_EINVAL;
  }
}

extern "C" size_t glamr_smpl_workspace_bytes(const glamr_smpl_t* m, int n) {
  if (!m || n < 0) return 0;
  return smpl_workspace_floats(n, m->dev.S) * sizeof(float);
}

extern "C" size_t glamr_smpl_fk_workspace_bytes(const glamr_smpl_t* m, int n) {
  if (!m || n < 0) return 0;
  return smpl_workspace_floats_fk(n, m->dev.S) * sizeof(float);
}

extern "C" int glamr_smpl_forward(const glamr_smpl_t* m, int n, const float* global_orient, const float* body_pose,
                                  const float* betas, const float* root_trans, const float* root_scale, int orig_joints,
                                  float* joints, float* vertices, void* workspace, size_t workspace_bytes, void* stream) {
  if (!m || n < 0 || !body_pose || !betas || !joints || !workspace) return GLAMR_EINVAL;
  if (workspace_bytes < glamr_smpl_workspace_bytes(m, n)) return GLAMR_ENOSPACE;
  if (n == 0) return GLAMR_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const SmplWorkspace w = smpl_carve_workspace(workspace, n, m->dev.S);
  int rc;
  if ((rc = launch_pose_prep(m->dev, n, global_orient, body_pose, betas, 1, w, s))) return rc;
  if ((rc = launch_lbs(m->dev, 0, n, betas, w, vertices, s))) return rc;
  if ((rc = launch_joints_finalize(m->dev, n, orig_joints, root_trans, root_scale, w, joints, s))) return rc;
  if (vertices && root_trans)
    if ((rc = launch_reroot_vertices(n, w.root_raw, root_trans, root_scale, vertices, s))) return rc;
  return GLAMR_OK;
}

extern "C" int glamr_smpl_fk24(const glamr_smpl_t* m, int n, const float* global_orient, const float* body_pose,
                               const float* root_trans, const float* root_scale, float* joints, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!m || n < 0 || !body_pose || !joints || !workspace) return GLAMR_EINVAL;
  if (workspace_bytes < glamr_smpl_fk_workspace_bytes(m, n)) return GLAMR_ENOSPACE;
  if (n == 0) return GLAMR_OK;
  cudaStream_t s = (cudaStream_t)stream;
  SmplWorkspace w = smpl_carve_workspace(workspace, n, m->dev.S);
  w.tcA = nullptr;                             // FK only: no blend features, no skinning operands
  w.skB = nullptr;
  w.vp_tiled = 0;
  int rc = launch_pose_prep(m->dev, n, global_orient, body_pose, nullptr, 0, w, s);
  if (rc) return rc;
  fk24_finalize_kernel<<<(n * kNJ * 3 + 255) / 256, 256, 0, s>>>(n, w.jposed, root_trans, root_scale, joints);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}
