// Device-resident SMPL constants, re-tiled for the kernels of smpl_kernels.cu (layout is documented in DESIGN.md).
#pragma once
#include "common.cuh"
#include "glamr_math.cuh"

namespace glamr {

struct SmplDev {
  // dense constants
  const float* pd_tiles;     // [54][207][384]  posedirs, vertex-tile major: one contiguous 13,824 B block per
                             //                 (tile, 9-row chunk) so a CTA streams its slab with 1-D bulk TMA
  const float* tcB;          // [81 col tiles][28 K chunks][hi | lo][2 K groups][256 cols][4]  the blend basis (posedirs | shapedirs |
                             //                 v_template) pre-split into tf32 hi / lo and pre-tiled as the UMMA K-major core-matrix image:
                             //                 one contiguous 16 KB block per (tile, chunk) = one bulk copy per pipeline stage
  const float* skW;          // [54 vertex tiles][hi | lo][6 joint groups][128 vertices][4]  dense skinning weights W[v][24], tf32 hi / lo,
                             //                 UMMA K-major image: one contiguous 24 KB block per vertex tile (lbs_skin_tc_kernel)
  const float* v_template;   // [6912][3]  (padded with zeros)
  const float* shapedirs;    // [6912][30] ([v][c][l] as in the model file)
  const float* j_template;   // [24][3]    J_regressor @ v_template
  const float* j_shapedirs;  // [24][3][10] J_regressor @ shapedirs   (J(beta) = j_template + j_shapedirs . beta)
  // K-sparse skinning weights (K = max non-zeros per vertex, rows zero-padded)
  const float* skin_w;       // [6912][K]
  const uint8_t* skin_j;     // [6912][K]
  int K;
  // vertices that feed a picked joint or an extra-regressor row ("support"), compacted
  const int32_t* compact_of_vertex;  // [6912] index into the support list or -1
  int S;                     // support size
  const int32_t* reg_ptr;    // [n_extra+1]  CSR over J_regressor_extra rows
  const int32_t* reg_ci;     // [nnz] compact vertex index
  const float* reg_w;        // [nnz]
  const int32_t* pick_ci;    // [n_picks] compact vertex index of each picked vertex
  const int32_t* joint_map;  // [n_map] into [24 | n_picks | n_extra]
  int n_extra, n_picks, n_map;
  int parents[kNJ];
  int level[kNJ];
  int n_levels;
};

struct SmplWorkspace {
  float* A;         // [n/32][24][32][12] relative joint transforms (3x4 row-major per joint), tile-major
  float* pf;        // [n/32][23][9][32] pose feature (R_j - I), j = 1..23, tile-major for bulk TMA (208 floats per frame reserved)
  float* jposed;    // [n][24][3]   posed LBS joints
  float* vcompact;  // [n][S][3]    skinned support vertices
  float* root_raw;  // [n][3]       un-rooted joint 0 (for vertex re-rooting)
  float* tcA;       // [n/128][28][hi | lo][2][128][4]  blend features (pose feature | betas | 1 | 0-pad), tf32 hi / lo, UMMA image per
                    //              (128-frame tile, K chunk): 8 KB contiguous = one bulk copy per stage
  float* vpT;       // [20736][mpad]  blended vertices v_posed, TRANSPOSED (column-major over frames) so that the skinning kernel's
                    //              lanes = frames read 128 contiguous bytes per vertex coordinate
  int mpad;         // frames padded to a multiple of 128
  float* skB;       // [ceil(mpad/20)][hi | lo][6 joint groups][20 frames x 12][4]  the relative joint transforms as the B operand of the
                    //              tensor-core skinning (row = frame-in-tile * 12 + element of the 3x4, K = joint), tf32 hi / lo
  int vp_tiled;     // 1: v_posed is stored frame-tiled for lbs_skin_tc_kernel: [ceil(mpad/20)][20736 cols][20 frames] (the 128 vertices x
                    //    20 frames of a skinning tile are one contiguous 30,720 B block = one bulk copy); 0: vpT as described above
};

// FK only (glamr_smpl_fk24): the kinematic-chain scratch without the blend operands (they are carved last)
inline size_t smpl_workspace_floats_fk(int n, int S) {
  const size_t n32 = ((size_t)n + 31) / 32 * 32;
  return (size_t)n * (kNJ * 3 + (size_t)S * 3 + 3) + n32 * (kPFPad + kNJ * 12) + 64 + 64;
}
inline size_t smpl_workspace_floats(int n, int S) {
  const size_t n32 = ((size_t)n + 31) / 32 * 32;   // the pose feature is tile-major over whole 32-frame tiles
  const size_t n128 = ((size_t)n + kTcM - 1) / kTcM * kTcM;
  return (size_t)n * (kNJ * 3 + (size_t)S * 3 + 3) + n32 * (kPFPad + kNJ * 12) + 64 + 64 +
         (n128 / kTcM) * kTcChunks * kTcAStageFloats + (size_t)kTcCols * ((n128 + kSkF - 1) / kSkF * kSkF) +
         ((n128 + kSkF - 1) / kSkF) * kSkBImageFloats + 64;
}
int lbs_path();                              // 2 tensor-core blend + tensor-core skinning, 1 tensor-core blend + SIMT skinning, 0 one-kernel FP32 SIMT path
inline SmplWorkspace smpl_carve_workspace(void* base, int n, int S) {
  SmplWorkspace w;
  float* p = (float*)base;
  w.A = p; p += ((size_t)n + 31) / 32 * 32 * kNJ * 12;
  w.pf = p; p += ((size_t)n + 31) / 32 * 32 * kPFPad;
  w.jposed = p; p += (size_t)n * kNJ * 3;
  w.vcompact = p; p += (size_t)n * S * 3;
  w.root_raw = p; p += (size_t)n * 3;
  p = (float*)(((uintptr_t)p + 255) & ~(uintptr_t)255);          // bulk-copy sources: 16-byte aligned (256 for good measure)
  w.mpad = (int)(((size_t)n + kTcM - 1) / kTcM * kTcM);
  w.tcA = p; p += (size_t)(w.mpad / kTcM) * kTcChunks * kTcAStageFloats;
  w.skB = p; p += (size_t)((w.mpad + kSkF - 1) / kSkF) * kSkBImageFloats;
  w.vpT = p;                                   // [20736][mpad] or, frame-tiled, [ceil(mpad/20)][20736][20]
  w.vp_tiled = lbs_path() == 2 ? 1 : 0;
  return w;
}

#if defined(__CUDACC__)
// un-rooted joint `idx` of [24 LBS | picks | extra regressed] for local frame-person f  (lib/models/smpl.py:299-301)
__device__ __forceinline__ void raw_joint(const SmplDev& m, const SmplWorkspace& w, int f, int idx, float* o) {
  if (idx < kNJ) {
    const float* p = w.jposed + ((size_t)f * kNJ + idx) * 3;
    o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
  } else if (idx < kNJ + m.n_picks) {
    const float* p = w.vcompact + ((size_t)f * m.S + m.pick_ci[idx - kNJ]) * 3;
    o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
  } else {
    const int r = idx - kNJ - m.n_picks;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    for (int e = m.reg_ptr[r]; e < m.reg_ptr[r + 1]; ++e) {
      const float* p = w.vcompact + ((size_t)f * m.S + m.reg_ci[e]) * 3;
      const float wt = m.reg_w[e];
      a0 = fmaf(wt, p[0], a0); a1 = fmaf(wt, p[1], a1); a2 = fmaf(wt, p[2], a2);
    }
    o[0] = a0; o[1] = a1; o[2] = a2;
  }
}

// One warp evaluates frame-person `f` (index into the workspace): lane j < 24 owns joint j.
//   R_j = rodrigues(pose_j)                                   lbs.py:446-477
//   J_j = j_template + j_shapedirs . beta  (== J_regressor @ v_shaped, lbs.py:240-244, by linearity)
//   G_j = G_parent(j) * [R_j | J_j - J_parent],  A_j = G_j - [0 | G_j J_j]      lbs.py:493-548
// orient3: 3 floats or nullptr (zeros); bp: this frame's 69 body-pose floats; beta: 10 floats or nullptr (template joints).
__device__ __forceinline__ void pose_prep_frame(const SmplDev& m, int f, const float* __restrict__ orient3, const float* __restrict__ bp,
                                                const float* __restrict__ beta, const SmplWorkspace& w, int lane) {
  const int j = lane < kNJ ? lane : kNJ - 1;
  float r[3];
  if (j == 0) {
    r[0] = orient3 ? orient3[0] : 0.0f;
    r[1] = orient3 ? orient3[1] : 0.0f;
    r[2] = orient3 ? orient3[2] : 0.0f;
  } else {
    const float* q = bp + (j - 1) * 3;
    r[0] = q[0]; r[1] = q[1]; r[2] = q[2];
  }
  float R[9];
  rodrigues_smplx(r, R);
  float J[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float v = m.j_template[j * 3 + c];
    if (beta) {
      const float* js = m.j_shapedirs + (j * 3 + c) * kNB;
#pragma unroll
      for (int l = 0; l < kNB; ++l) v = fmaf(js[l], beta[l], v);
    }
    J[c] = v;
  }
  if (lane >= 1 && lane < kNJ) {
    // pose feature (R_j - I), stored tile-major [n/32][chunk = j-1][k][n%32] so the LBS kernel fetches a CTA's
    // [9 x 32] chunk with one bulk copy
    float* pf = w.pf + (((size_t)(f >> 5) * kNChunks + (lane - 1)) * kChunkK) * 32 + (f & 31);
#pragma unroll
    for (int k = 0; k < 9; ++k) pf[k * 32] = R[k] - ((k % 4 == 0) ? 1.0f : 0.0f);
  }
  if (w.tcA) {
    // the same features (+ betas, + the constant 1 that multiplies v_template, + zero padding) as the A operand of the
    // tensor-core blend GEMM: tf32 hi / lo, K-major core-matrix image of this frame's 128-frame tile
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
#pragma unroll
      for (int k = 0; k < 9; ++k) put((lane - 1) * 9 + k, R[k] - ((k % 4 == 0) ? 1.0f : 0.0f));
    } else if (lane == 0) {
#pragma unroll
      for (int l = 0; l < kNB; ++l) put(kPF + l, beta ? beta[l] : 0.0f);
      put(kPF + kNB, 1.0f);
#pragma unroll
      for (int k = kTcFeat; k < kTcK; ++k) put(k, 0.0f);
    }
  }

  float GR[9], Gt[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) GR[k] = R[k];
#pragma unroll
  for (int k = 0; k < 3; ++k) Gt[k] = J[k];
  const int par = m.parents[j] < 0 ? 0 : m.parents[j];
  const int lev = m.level[j];
  for (int l = 1; l < m.n_levels; ++l) {
    float pR[9], pt[3], pJ[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) pR[k] = __shfl_sync(0xffffffffu, GR[k], par);
#pragma unroll
    for (int k = 0; k < 3; ++k) pt[k] = __shfl_sync(0xffffffffu, Gt[k], par);
#pragma unroll
    for (int k = 0; k < 3; ++k) pJ[k] = __shfl_sync(0xffffffffu, J[k], par);
    if (lev == l) {
      float nR[9], rel[3], nt[3];
      mat3_mul(pR, R, nR);
      rel[0] = J[0] - pJ[0]; rel[1] = J[1] - pJ[1]; rel[2] = J[2] - pJ[2];
      mat3_vec(pR, rel, nt);
#pragma unroll
      for (int k = 0; k < 9; ++k) GR[k] = nR[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) Gt[k] = nt[k] + pt[k];
    }
  }
  if (lane < kNJ) {
    float* jp = w.jposed + ((size_t)f * kNJ + j) * 3;
    jp[0] = Gt[0]; jp[1] = Gt[1]; jp[2] = Gt[2];
    float GJ[3];
    mat3_vec(GR, J, GJ);
    // A_j (3x4 row-major, 12 floats) stored tile-major: [n/32][j][n%32][12], so the LBS kernel fetches a CTA's
    // [24][32][12] tile with one bulk copy and a lane (= frame) reads its 12 floats with three LDS.128 (48-byte lane
    // stride: the 8 lanes of a quarter warp hit 8 distinct 16-byte bank groups)
    float4* A = reinterpret_cast<float4*>(w.A + (((size_t)(f >> 5) * kNJ + j) * 32 + (f & 31)) * 12);
#pragma unroll
    for (int i = 0; i < 3; ++i) A[i] = make_float4(GR[i * 3 + 0], GR[i * 3 + 1], GR[i * 3 + 2], Gt[i] - GJ[i]);
    if (w.vp_tiled) {
      // the same 12 numbers as column j of the tensor-core skinning's B operand: row = frame-in-tile * 12 + element
      float* img = w.skB + (size_t)(f / kSkF) * kSkBImageFloats + ((size_t)(j >> 2) * kSkN + (f % kSkF) * 12) * 4 + (j & 3);
#pragma unroll
      for (int i = 0; i < 12; ++i) {
        const float v = (i & 3) < 3 ? GR[(i >> 2) * 3 + (i & 3)] : Gt[i >> 2] - GJ[i >> 2];
        float hi, lo;
        split_tf32(v, hi, lo);
        img[i * 4] = hi;
        img[kSkBHalf + i * 4] = lo;
      }
    }
  }
}
#endif

// launches (smpl_kernels.cu); all asynchronous on `s`
// orient may be NULL (zeros).  use_betas == 0 -> rest joints from the template only (SMPL.get_joints).
int launch_pose_prep(const SmplDev& m, int n, const float* orient, const float* body_pose, const float* betas,
                     int use_betas, const SmplWorkspace& w, cudaStream_t s);
// n_begin..n_end: frame-person range to skin.  vertices may be NULL.
int launch_lbs(const SmplDev& m, int n_begin, int n_end, const float* betas, const SmplWorkspace& w, float* vertices,
               cudaStream_t s);
// tensor-core path in parts (the optimiser pipelines them: the blend depends on body pose / betas only):
// blend = features (the GEMM's A operand) + GEMM; the skinning reads the blend's v_posed
int launch_blend_features(int n, const float* body_pose, const float* betas, const SmplWorkspace& w, cudaStream_t s);
int launch_blend_gemm(const SmplDev& m, int n, const SmplWorkspace& w, cudaStream_t s);
int launch_blend(const SmplDev& m, int n, const float* body_pose, const float* betas, const SmplWorkspace& w, cudaStream_t s);
int launch_skin(const SmplDev& m, int n, const SmplWorkspace& w, float* vertices, cudaStream_t s);
int lbs_kernel_count(const SmplDev& m);      // kernels one launch_lbs call launches
int launch_joints_finalize(const SmplDev& m, int n, int orig_joints, const float* root_trans, const float* root_scale,
                           const SmplWorkspace& w, float* joints, cudaStream_t s);
int launch_reroot_vertices(int n, const float* root_raw, const float* root_trans, const float* root_scale,
                           float* vertices, cudaStream_t s);

}  // namespace glamr

struct glamr_smpl {
  glamr::SmplDev dev;
  void* allocs[16];
  int n_allocs;
};
