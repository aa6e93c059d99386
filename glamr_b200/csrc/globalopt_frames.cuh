// Per-frame forward / residual / backward "frame functions" of one global-optimisation iteration.  The CUDA
// kernels in globalopt_kernels.cu call them with one thread per frame (or frame-person) and supply the prefix
// scans between phases; tests/host_harness runs the very same functions sequentially with g++ so the analytic
// backward can be checked against torch autograd of the oracle on the GPU-less build box.
//
// What is computed follows global_recon/models/global_recon_model.py:394-531 (forward),
// traj_pred/utils/traj_utils.py:65-88 (trajectory codec), global_recon/models/loss_func.py (residuals); the
// backward is the hand-derived reverse of exactly those formulas (SURVEY.md Appendix A.5-A.6).
#pragma once
#include "glamr_math.cuh"
#include "../../include/glamr_b200.h"

namespace glamr {

constexpr float kFps = 30.0f;
constexpr float kFps2 = 900.0f;

struct OptScratch {
  float* heading;       // [N]     d_heading, then (after the scan) heading, local frames of each person
  float* xy;            // [N][2]  world-frame d_xy, then (after the scan) xy
  float* traj_local;    // [N][11]
  float* orient_base;   // [N][3]
  float* trans_base;    // [N][3]
  float* orient_world;  // [N][3]
  float* trans_world;   // [N][3]
  float* cam;           // [T][12] world->cam (3x4 row-major)
  float* cam_inv;       // [T][12]
  float* cam_d6;        // [T][6]  6d of cam_inv rotation incl. residual (mode 3)
  float* joints_world;  // [N][J][3]
  float* kp_pred;       // [N][J][2]
  float* orient_ciw;    // [N][3]  smpl_orient_cam_in_world
  float* trans_ciw;     // [N][3]  root_trans_cam_in_world
  float* g_orient;      // [N][3]  dL/d smpl_orient_world
  float* g_trans;       // [N][3]  dL/d root_trans_world
  float* g_cam;         // [N][12] per frame-person dL/d cam (R 9, t 3)
  float* g_cam_fix;     // [T][12] per-frame dL/d (cam_rot_6d, cam_trans) [9 used] in fixed-camera mode; mode 3: dL/d(mean cam_inv)
  float* g_xy;          // [N][2]  backward scan buffer
  float* g_head;        // [N]
  float* grad;          // [n_params]
};

struct OptCtx {
  glamr_problem_t pb;
  OptScratch sc;
  const float* theta;
  float gs[GLAMR_NUM_TERMS];   // weight / normaliser for terms that enter the total, else 0
};

struct TermAcc {
  double v[GLAMR_NUM_TERMS];
  GLAMR_HD void clear() {
    for (int k = 0; k < GLAMR_NUM_TERMS; ++k) v[k] = 0.0;
  }
};

GLAMR_HD void mat34_inverse(const float* M, float* I) {
  // lib/utils/torch_transform.py:274-279  [R^T | -R^T t]
  I[0] = M[0]; I[1] = M[4]; I[2] = M[8];
  I[4] = M[1]; I[5] = M[5]; I[6] = M[9];
  I[8] = M[2]; I[9] = M[6]; I[10] = M[10];
  I[3] = -(M[0] * M[3] + M[4] * M[7] + M[8] * M[11]);
  I[7] = -(M[1] * M[3] + M[5] * M[7] + M[9] * M[11]);
  I[11] = -(M[2] * M[3] + M[6] * M[7] + M[10] * M[11]);
}
GLAMR_HD void mat34_R(const float* M, float* R) {
  R[0] = M[0]; R[1] = M[1]; R[2] = M[2]; R[3] = M[4]; R[4] = M[5]; R[5] = M[6]; R[6] = M[8]; R[7] = M[9]; R[8] = M[10];
}

// ------------------------------------------------------------------------------------------------ trajectory fwd
// global_recon_model.py:394-419 + traj_utils.py:65-70: per local frame i of person p.
// values only: tl[11] = traj_local row of local frame i, returns the (re-wrapped) heading increment that enters the scan
GLAMR_HD float traj_pre_vals(const OptCtx& c, int p, int i, float* tl) {
  const glamr_person_t& ps = c.pb.persons[p];
  const float* pr = ps.traj_local_pred + (size_t)i * 11;
  const float* th = c.theta;
  float h = safe_atan2(pr[10], pr[9]);
  if (i == 0) {
    h += th[ps.off_heading];
    tl[0] = pr[0] + th[ps.off_xy];
    tl[1] = pr[1] + th[ps.off_xy + 1];
  } else {
    h += th[ps.off_dheading + i - 1] * ps.dheading_mask[i - 1];
    tl[0] = pr[0] + th[ps.off_dxy + 2 * (i - 1)];
    tl[1] = pr[1] + th[ps.off_dxy + 2 * (i - 1) + 1];
  }
  tl[2] = pr[2] + th[ps.off_z + i];
  const float rm = ps.rot_mask ? ps.rot_mask[i] : 1.0f;
#pragma unroll
  for (int k = 0; k < 6; ++k) tl[3 + k] = pr[3 + k] + th[ps.off_rot + 6 * i + k] * rm;
  const float ch = cosf(h), sh = sinf(h);
  tl[9] = ch;
  tl[10] = sh;
  return safe_atan2(sh, ch);
}
GLAMR_HD void traj_pre(const OptCtx& c, int p, int i) {
  const int n = p * c.pb.T + c.pb.persons[p].start + i;
  float tl[11];
  c.sc.heading[n] = traj_pre_vals(c, p, i, tl);
#pragma unroll
  for (int k = 0; k < 11; ++k) c.sc.traj_local[(size_t)n * 11 + k] = tl[k];
}
// after the inclusive scan of heading: rotate d_xy of frame i >= 1 by heading[i-1]   (traj_utils.py:76-77)
GLAMR_HD void traj_mid(const OptCtx& c, int p, int i) {
  const glamr_person_t& ps = c.pb.persons[p];
  const int n = p * c.pb.T + ps.start + i;
  const float* tl = c.sc.traj_local + (size_t)n * 11;
  float x = tl[0], y = tl[1];
  if (i > 0) {
    const float t = c.sc.heading[n - 1];
    const float ct = cosf(t), st = sinf(t);
    const float rx = x * ct - y * st, ry = x * st + y * ct;
    x = rx; y = ry;
  }
  c.sc.xy[2 * (size_t)n] = x;
  c.sc.xy[2 * (size_t)n + 1] = y;
}
// after the inclusive scan of xy: world pose of absolute frame t  (traj_utils.py:78-88, global_recon_model.py:421-470)
GLAMR_HD void local_quat(const float* d6, float heading, float* q_hl, float* local_q, float* hq) {
  float R[9];
  rot6d_to_rotmat(d6, R);
  rotmat_to_quat(R, local_q);
  const float ha[3] = {0.0f, 0.0f, heading};
  aa_to_quat(ha, hq);
  quat_mul(hq, local_q, q_hl);
}
// world pose of absolute frame t from its traj_local row `tl`, scanned heading and scanned xy (ignored outside the exist range);
// writes orient/trans base + world of frame-person n, returns nothing else
GLAMR_HD void traj_post_vals(const OptCtx& c, int p, int t, const float* tl, float heading, float x, float y, float* ow_out) {
  const glamr_person_t& ps = c.pb.persons[p];
  const int T = c.pb.T;
  const int n = p * T + t;
  const int i = t - ps.start;
  float ob[3], tb[3];
  if (i >= 0 && i < ps.len) {
    float q_hl[4], lq[4], hq[4], q[4];
    local_quat(tl + 3, heading, q_hl, lq, hq);
    const float base[4] = {0.5f, 0.5f, 0.5f, 0.5f};
    quat_mul(q_hl, base, q);
    quat_to_aa(q, ob);
    tb[0] = x; tb[1] = y; tb[2] = tl[2];
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) { ob[k] = ps.orient_base_init[t * 3 + k]; tb[k] = ps.trans_base_init[t * 3 + k]; }
  }
  float ow[3], tw[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { ow[k] = ob[k]; tw[k] = tb[k]; }
  if (c.pb.use_world_res) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      ow[k] += c.theta[ps.off_orient_res + t * 3 + k];
      tw[k] += c.theta[ps.off_trans_res + t * 3 + k];
    }
  }
  if (c.pb.has_world_dheading) {
    const float da[3] = {0.0f, 0.0f, c.theta[ps.off_world_dheading + t]};
    float dq[4], bq[4], q[4];
    aa_to_quat(da, dq);
    aa_to_quat(ob, bq);
    quat_mul(dq, bq, q);
    quat_to_aa(q, ow);
#pragma unroll
    for (int k = 0; k < 3; ++k) tw[k] = tb[k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    c.sc.orient_base[(size_t)n * 3 + k] = ob[k];
    c.sc.trans_base[(size_t)n * 3 + k] = tb[k];
    c.sc.orient_world[(size_t)n * 3 + k] = ow[k];
    c.sc.trans_world[(size_t)n * 3 + k] = tw[k];
    if (ow_out) ow_out[k] = ow[k];
  }
}
GLAMR_HD void traj_post(const OptCtx& c, int p, int t) {
  const glamr_person_t& ps = c.pb.persons[p];
  const int n = p * c.pb.T + t;
  const int i = t - ps.start;
  float* tl = c.sc.traj_local + (size_t)n * 11;
  if (i >= 0 && i < ps.len) {
    traj_post_vals(c, p, t, tl, c.sc.heading[n], c.sc.xy[2 * (size_t)n], c.sc.xy[2 * (size_t)n + 1], nullptr);
  } else {
    for (int k = 0; k < 11; ++k) tl[k] = 0.0f;
    traj_post_vals(c, p, t, tl, 0.0f, 0.0f, 0.0f, nullptr);
  }
}

// ------------------------------------------------------------------------------------------------ camera fwd
// global_recon_model.py:473-508.  cam[t] is world->cam, cam_inv[t] its inverse.
GLAMR_HD void person_world_transform(const OptCtx& c, int p, int t, float* M) {
  // person_transform_world = make_transform(smpl_orient_world, root_trans_world)  (:470)
  const size_t n = (size_t)p * c.pb.T + t;
  float R[9];
  aa_to_rotmat(c.sc.orient_world + n * 3, R);
  M[0] = R[0]; M[1] = R[1]; M[2] = R[2]; M[3] = c.sc.trans_world[n * 3 + 0];
  M[4] = R[3]; M[5] = R[4]; M[6] = R[5]; M[7] = c.sc.trans_world[n * 3 + 1];
  M[8] = R[6]; M[9] = R[7]; M[10] = R[8]; M[11] = c.sc.trans_world[n * 3 + 2];
}
GLAMR_HD void mat34_mul(const float* A, const float* B, float* o) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v = A[i * 4] * B[j] + A[i * 4 + 1] * B[4 + j] + A[i * 4 + 2] * B[8 + j];
      if (j == 3) v += A[i * 4 + 3];
      o[i * 4 + j] = v;
    }
  }
}
// person2cam of frame s, corrected by the person's residual variables when it has them:
// person2cam @ make_transform(person2cam_res_rot, person2cam_res_trans, '6d')  (:484-488).  Returns the 3x4 to use
// (the constant table itself, or `buf`).
GLAMR_HD const float* person2cam_at(const OptCtx& c, const glamr_person_t& ps, int s, float* buf) {
  const float* P2C = ps.person2cam + (size_t)s * 12;
  if (ps.off_person2cam_res < 0) return P2C;
  const float* tr = c.theta + ps.off_person2cam_res + 6 * c.pb.T + 3 * s;
  float R[9];
  rot6d_to_rotmat(c.theta + ps.off_person2cam_res + 6 * s, R);
  const float B[12] = {R[0], R[1], R[2], tr[0], R[3], R[4], R[5], tr[1], R[6], R[7], R[8], tr[2]};
  mat34_mul(P2C, B, buf);
  return buf;
}
// mean over visible persons of person_transform_world @ person2cam at source frame s  (:482-492)
GLAMR_HD void mean_cam_inv(const OptCtx& c, int s, float* M) {
#pragma unroll
  for (int k = 0; k < 12; ++k) M[k] = 0.0f;
  for (int p = 0; p < c.pb.P; ++p) {
    const glamr_person_t& ps = c.pb.persons[p];
    if (ps.vis[s] == 0.0f) continue;
    float Tw[12], C[12], P2C[12];
    person_world_transform(c, p, s, Tw);
    mat34_mul(Tw, person2cam_at(c, ps, s, P2C), C);
#pragma unroll
    for (int k = 0; k < 12; ++k) M[k] += C[k];
  }
  const float inv = c.pb.inv_num_persons[s];
#pragma unroll
  for (int k = 0; k < 12; ++k) M[k] *= inv;
}
GLAMR_HD void cam_forward(const OptCtx& c, int t) {
  float cam[12], inv[12];
  const int mode = c.pb.cam_mode;
  if (mode == GLAMR_CAM_CONST) {
#pragma unroll
    for (int k = 0; k < 12; ++k) cam[k] = c.pb.cam_pose_const[(size_t)t * 12 + k];
    mat34_inverse(cam, inv);
  } else if (mode == GLAMR_CAM_PER_FRAME || mode == GLAMR_CAM_FIXED) {
    const int r = (mode == GLAMR_CAM_FIXED) ? 0 : t;
    float R[9];
    rot6d_to_rotmat(c.theta + c.pb.off_cam_rot + 6 * r, R);
    const float* tc = c.theta + c.pb.off_cam_trans + 3 * r;
    cam[0] = R[0]; cam[1] = R[1]; cam[2] = R[2]; cam[3] = tc[0];
    cam[4] = R[3]; cam[5] = R[4]; cam[6] = R[5]; cam[7] = tc[1];
    cam[8] = R[6]; cam[9] = R[7]; cam[10] = R[8]; cam[11] = tc[2];
    mat34_inverse(cam, inv);
  } else {
    float M[12], R[9], d6[6];
    mean_cam_inv(c, c.pb.fill_src[t], M);
    mat34_R(M, R);
    rotmat_to_rot6d(R, d6);
    const int e = c.pb.empty_index[t];
    if (e >= 0) {
#pragma unroll
      for (int k = 0; k < 6; ++k) d6[k] += c.theta[c.pb.off_cam_rot + 6 * e + k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) c.sc.cam_d6[(size_t)t * 6 + k] = d6[k];
    rot6d_to_rotmat(d6, R);
    float tt[3] = {M[3], M[7], M[11]};
    if (c.pb.trans_res_all) {
#pragma unroll
      for (int k = 0; k < 3; ++k) tt[k] += c.theta[c.pb.off_cam_trans + 3 * t + k];
    } else if (e >= 0) {
#pragma unroll
      for (int k = 0; k < 3; ++k) tt[k] += c.theta[c.pb.off_cam_trans + 3 * e + k];
    }
    inv[0] = R[0]; inv[1] = R[1]; inv[2] = R[2]; inv[3] = tt[0];
    inv[4] = R[3]; inv[5] = R[4]; inv[6] = R[5]; inv[7] = tt[1];
    inv[8] = R[6]; inv[9] = R[7]; inv[10] = R[8]; inv[11] = tt[2];
    mat34_inverse(inv, cam);
  }
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    c.sc.cam[(size_t)t * 12 + k] = cam[k];
    c.sc.cam_inv[(size_t)t * 12 + k] = inv[k];
  }
}

// ------------------------------------------------------------------------------------------------ frame residuals
// Per frame-person (p,t): projection + kp_2d (+dist), cam_traj_rot/trans, traj rot/trans smoothness, rel_transform.
// Writes kp_pred, orient_ciw, trans_ciw, g_orient, g_trans, g_cam and adds un-normalised sums to `acc`.
// The SMPL dependence is handled through the rigid form  joints = R(orient) b_k + trans  (b_k body-frame offsets,
// constant w.r.t. the optimisation variables; SURVEY.md §0.5): dL/dR = sum_k g_k (R^T (joint_k - trans))^T.
// Contribution of joint k of frame-person (p,t) to the reprojection terms (loss_func.py:15-57, geometry.py:23-25) and to
// the gradients w.r.t. camera (g_Rc, g_tc), translation (g_tw) and the SMPL root rotation matrix (g_Rs).  The CUDA kernel
// runs one lane per joint and sums these with warp shuffles; the host harness loops over k.
struct KpGrad {
  float g_tc[3], g_Rc[9], g_tw[3], g_Rs[9];
  double kp, dist;
  GLAMR_HD void clear() {
    for (int i = 0; i < 3; ++i) { g_tc[i] = 0.0f; g_tw[i] = 0.0f; }
    for (int i = 0; i < 9; ++i) { g_Rc[i] = 0.0f; g_Rs[i] = 0.0f; }
    kp = 0.0; dist = 0.0;
  }
};
GLAMR_HD void kp_joint_terms(const OptCtx& c, int p, int t, int k, const float* jw, const float* Rc, const float* tc, const float* Rs,
                             const float* tw, KpGrad& o) {
  const glamr_person_t& ps = c.pb.persons[p];
  const int J = c.pb.J;
  const size_t n = (size_t)p * c.pb.T + t;
  const float* K = ps.cam_K + (size_t)t * 9;
  const float gsk = c.gs[GLAMR_T_KP_2D];
  float Xc[3], uv[2];
  mat3_vec(Rc, jw, Xc);
  Xc[0] += tc[0]; Xc[1] += tc[1]; Xc[2] += tc[2];
  project(K, Xc, uv);
  c.sc.kp_pred[(n * J + k) * 2] = uv[0];
  c.sc.kp_pred[(n * J + k) * 2 + 1] = uv[1];
  const float dx = uv[0] - ps.kp_target[((size_t)t * J + k) * 2];
  const float dy = uv[1] - ps.kp_target[((size_t)t * J + k) * 2 + 1];
  const float wk = ps.kp_w[(size_t)t * J + k];
  const float dm = ps.kp_dist_mask[(size_t)t * J + k];
  if (dm != 0.0f) o.dist += (double)(dm * sqrtf(dx * dx + dy * dy));
  if (wk != 0.0f) {
    o.kp += (double)wk * ((double)gmof(dx) + (double)gmof(dy));
    if (gsk != 0.0f) {
      const float guv[2] = {gsk * wk * gmof_grad(dx), gsk * wk * gmof_grad(dy)};
      float gX[3], gj[3], b[3], d[3];
      project_vjp(K, Xc, guv, gX);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        o.g_tc[a] += gX[a];
#pragma unroll
        for (int bb = 0; bb < 3; ++bb) o.g_Rc[a * 3 + bb] += gX[a] * jw[bb];
      }
      mat3_tvec(Rc, gX, gj);
      d[0] = jw[0] - tw[0]; d[1] = jw[1] - tw[1]; d[2] = jw[2] - tw[2];
      mat3_tvec(Rs, d, b);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        o.g_tw[a] += gj[a];
#pragma unroll
        for (int bb = 0; bb < 3; ++bb) o.g_Rs[a * 3 + bb] += gj[a] * b[bb];
      }
    }
  }
}

// quat_angle_diff(a, b) (lib/utils/torch_transform.py:48-60): angle = acos(clamp(2 w^2 - 1, -1 + 1e-6, 1 - 1e-6)) with w the scalar part
// of a (x) conj(b), i.e. the dot product of the two quaternions; also d(angle)/d(w) (0 where the clamp is active).
GLAMR_HD void quat_angle_dot(const float* a, const float* b, float& angle, float& dangle_dw) {
  // Near-identical rotations sit at the clamp, where acos amplifies the last bits of w: in float32 the angle of consecutive frames
  // carries ~0.5 % noise in ANY evaluation order (the reference's own float32 value is 0.3 % off its float64 value on the test
  // tracks); the plain dot product is the most accurate form.
  const float w = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3];
  const float u = 2.0f * w * w - 1.0f;
  const float lo = -1.0f + 1e-6f, hi = 1.0f - 1e-6f;
  const float uc = fminf(fmaxf(u, lo), hi);
  angle = acosf(uc);
  dangle_dw = (u > lo && u < hi) ? -4.0f * w / sqrtf(1.0f - uc * uc) : 0.0f;
}

// Everything of frame-person (p,t) that is not per joint, given the summed joint contributions `kg`.
// section time stamps of one warp (tools/frame_sections.py): experiment build, device code only
#if defined(GLAMR_EXPERIMENT) && defined(__CUDACC__)
__device__ long long g_frame_stamps[2][16];
#endif
#if defined(GLAMR_EXPERIMENT) && defined(__CUDA_ARCH__)
#define GLAMR_STAMP(i) do { if (blockIdx.x == 0 || blockIdx.x == 37) if ((threadIdx.x & 127) == 0) g_frame_stamps[blockIdx.x != 0][i] = clock64(); } while (0)
#else
#define GLAMR_STAMP(i) do { } while (0)
#endif

GLAMR_HD void frame_rest(const OptCtx& c, int p, int t, const KpGrad& kg, TermAcc& acc) {
  GLAMR_STAMP(4);
  const glamr_problem_t& pb = c.pb;
  const glamr_person_t& ps = pb.persons[p];
  const int T = pb.T;
  const size_t n = (size_t)p * T + t;
  const float* ow = c.sc.orient_world + n * 3;
  const float* tw = c.sc.trans_world + n * 3;
  float Rc[9], tc[3];
  mat34_R(c.sc.cam + (size_t)t * 12, Rc);
  tc[0] = c.sc.cam[(size_t)t * 12 + 3]; tc[1] = c.sc.cam[(size_t)t * 12 + 7]; tc[2] = c.sc.cam[(size_t)t * 12 + 11];
  float g_ow[3] = {0, 0, 0}, g_tw[3], g_Rc[9], g_tc[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { g_tw[k] = kg.g_tw[k]; g_tc[k] = kg.g_tc[k]; }
#pragma unroll
  for (int k = 0; k < 9; ++k) g_Rc[k] = kg.g_Rc[k];
  acc.v[GLAMR_T_KP_2D] += kg.kp;
  acc.v[GLAMR_T_KP_2D_DIST] += kg.dist;
  if (c.gs[GLAMR_T_KP_2D] != 0.0f) {
    float g[3];
    rodrigues_smplx_vjp(ow, kg.g_Rs, g);
    g_ow[0] += g[0]; g_ow[1] += g[1]; g_ow[2] += g[2];
  }

  GLAMR_STAMP(5);
  // ---- camera-frame pose of the person + cam_traj_rot / cam_traj_trans (global_recon_model.py:512-513, loss_func.py:147-186)
  float Rw[9];
  aa_to_rotmat(ow, Rw);
  {
    float M[9], a[3];
    mat3_mul(Rc, Rw, M);
    rotmat_to_aa(M, a);
    float tcw[3];
    mat3_vec(Rc, tw, tcw);
    tcw[0] += tc[0]; tcw[1] += tc[1]; tcw[2] += tc[2];
#pragma unroll
    for (int k = 0; k < 3; ++k) { c.sc.orient_ciw[n * 3 + k] = a[k]; c.sc.trans_ciw[n * 3 + k] = tcw[k]; }
    const float wr = ps.ctr_w[t];
    if (wr != 0.0f && pb.cam_traj_rot_quat) {
      // rot_type 'quat' (loss_func.py:158-161): diff = quat_angle_diff(q(smpl_orient_cam), q(smpl_orient_cam_in_world))
      float q1[4], dd, dw;
      aa_to_quat(a, q1);
      const float* qt = ps.orient_cam_q + (size_t)t * 4;
      quat_angle_dot(qt, q1, dd, dw);
      acc.v[GLAMR_T_CAM_TRAJ_ROT] += (double)(wr * dd * dd);
      const float gsr = c.gs[GLAMR_T_CAM_TRAJ_ROT];
      if (gsr != 0.0f) {
        const float gw = 2.0f * gsr * wr * dd * dw;          // dL/d(dot)
        const float gq[4] = {gw * qt[0], gw * qt[1], gw * qt[2], gw * qt[3]};
        float ga[3], gM[9], t1[9], gRw[9], g[3];
        aa_to_quat_vjp(a, gq, ga);
        rotmat_to_aa_vjp(M, ga, gM);
        mat3_mult(gM, Rw, t1);        // dL/dRc = gM Rw^T
#pragma unroll
        for (int k = 0; k < 9; ++k) g_Rc[k] += t1[k];
        mat3_tmul(Rc, gM, gRw);       // dL/dRw = Rc^T gM
        aa_to_rotmat_vjp(ow, gRw, g);
        g_ow[0] += g[0]; g_ow[1] += g[1]; g_ow[2] += g[2];
      }
    } else if (wr != 0.0f) {
      float Ra[9], r6[6], diff[6];
      aa_to_rotmat(a, Ra);
      rotmat_to_rot6d(Ra, r6);
      float ss = 0.0f;
#pragma unroll
      for (int k = 0; k < 6; ++k) { diff[k] = ps.orient_cam_6d[(size_t)t * 6 + k] - r6[k]; ss += diff[k] * diff[k]; }
      acc.v[GLAMR_T_CAM_TRAJ_ROT] += (double)(wr * ss);
      const float gsr = c.gs[GLAMR_T_CAM_TRAJ_ROT];
      if (gsr != 0.0f) {
        float g6[6], gRa[9], ga[3], gM[9], t1[9], gRw[9], g[3];
#pragma unroll
        for (int k = 0; k < 6; ++k) g6[k] = -2.0f * gsr * wr * diff[k];
        rotmat_to_rot6d_vjp(g6, gRa);
        aa_to_rotmat_vjp(a, gRa, ga);
        rotmat_to_aa_vjp(M, ga, gM);
        mat3_mult(gM, Rw, t1);        // dL/dRc = gM Rw^T
#pragma unroll
        for (int k = 0; k < 9; ++k) g_Rc[k] += t1[k];
        mat3_tmul(Rc, gM, gRw);       // dL/dRw = Rc^T gM
        aa_to_rotmat_vjp(ow, gRw, g);
        g_ow[0] += g[0]; g_ow[1] += g[1]; g_ow[2] += g[2];
      }
    }
    const float wt = ps.ctt_w[t];
    if (wt != 0.0f) {
      float d[3], ss = 0.0f;
#pragma unroll
      for (int k = 0; k < 3; ++k) { d[k] = tcw[k] - ps.trans_cam[(size_t)t * 3 + k]; ss += d[k] * d[k]; }
      acc.v[GLAMR_T_CAM_TRAJ_TRANS] += (double)(wt * ss);
      const float gst = c.gs[GLAMR_T_CAM_TRAJ_TRANS];
      if (gst != 0.0f) {
        float g[3], gw[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) g[k] = 2.0f * gst * wt * d[k];
        mat3_tvec(Rc, g, gw);
#pragma unroll
        for (int a2 = 0; a2 < 3; ++a2) {
          g_tc[a2] += g[a2];
          g_tw[a2] += gw[a2];
#pragma unroll
          for (int b2 = 0; b2 < 3; ++b2) g_Rc[a2 * 3 + b2] += g[a2] * tw[b2];
        }
      }
    }
  }

  GLAMR_STAMP(6);
  float g_Rw[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  bool any_Rw = false;
  // ---- trajectory smoothness over ALL frames of the person (loss_func.py:117-144)
  if (pb.term_enabled[GLAMR_T_TRAJ_ROT_SMOOTH] && pb.traj_rot_smooth_quat) {
    // rot_type 'quat' (loss_func.py:126-128): (30 * quat_angle_diff(q[t+1], q[t]))^2 per frame pair
    const float gsm = c.gs[GLAMR_T_TRAJ_ROT_SMOOTH];
    float q0[4], gq[4] = {0, 0, 0, 0};
    aa_to_quat(ow, q0);
    if (t + 1 < T) {
      float qn[4], dd, dw;
      aa_to_quat(ow + 3, qn);
      quat_angle_dot(qn, q0, dd, dw);
      acc.v[GLAMR_T_TRAJ_ROT_SMOOTH] += (double)(kFps2 * dd * dd);
      const float gw = 2.0f * kFps2 * gsm * dd * dw;
#pragma unroll
      for (int k = 0; k < 4; ++k) gq[k] += gw * qn[k];
    }
    if (t > 0) {
      float qp[4], dd, dw;
      aa_to_quat(ow - 3, qp);
      quat_angle_dot(q0, qp, dd, dw);
      const float gw = 2.0f * kFps2 * gsm * dd * dw;
#pragma unroll
      for (int k = 0; k < 4; ++k) gq[k] += gw * qp[k];
    }
    if (gsm != 0.0f) {
      float g[3];
      aa_to_quat_vjp(ow, gq, g);
      g_ow[0] += g[0]; g_ow[1] += g[1]; g_ow[2] += g[2];
    }
  } else if (pb.term_enabled[GLAMR_T_TRAJ_ROT_SMOOTH]) {
    float r6[6], rp[6], rn[6], R2[9];
    rotmat_to_rot6d(Rw, r6);
    float g6[6] = {0, 0, 0, 0, 0, 0};
    const float gsm = c.gs[GLAMR_T_TRAJ_ROT_SMOOTH];
    if (t + 1 < T) {
      aa_to_rotmat(ow + 3, R2);
      rotmat_to_rot6d(R2, rn);
      float ss = 0.0f;
#pragma unroll
      for (int k = 0; k < 6; ++k) { const float d = rn[k] - r6[k]; ss += d * d; g6[k] -= 2.0f * kFps2 * gsm * d; }
      acc.v[GLAMR_T_TRAJ_ROT_SMOOTH] += (double)(kFps2 * ss);
    }
    if (t > 0) {
      aa_to_rotmat(ow - 3, R2);
      rotmat_to_rot6d(R2, rp);
#pragma unroll
      for (int k = 0; k < 6; ++k) g6[k] += 2.0f * kFps2 * gsm * (r6[k] - rp[k]);
    }
    if (gsm != 0.0f) {
      float gR[9];
      rotmat_to_rot6d_vjp(g6, gR);
#pragma unroll
      for (int k = 0; k < 9; ++k) g_Rw[k] += gR[k];
      any_Rw = true;
    }
  }
  if (pb.term_enabled[GLAMR_T_TRAJ_TRANS_SMOOTH]) {
    const float gsm = c.gs[GLAMR_T_TRAJ_TRANS_SMOOTH];
    if (t + 1 < T) {
      float ss = 0.0f;
#pragma unroll
      for (int k = 0; k < 3; ++k) { const float d = tw[3 + k] - tw[k]; ss += d * d; g_tw[k] -= 2.0f * kFps2 * gsm * d; }
      acc.v[GLAMR_T_TRAJ_TRANS_SMOOTH] += (double)(kFps2 * ss);
    }
    if (t > 0) {
#pragma unroll
      for (int k = 0; k < 3; ++k) g_tw[k] += 2.0f * kFps2 * gsm * (tw[k] - tw[k - 3]);
    }
  }

  GLAMR_STAMP(7);
  // ---- relative transforms between persons (loss_func.py:248-271): W_ij = inv(T_i) T_j against C_ij
  if (pb.rel_target && pb.term_enabled[GLAMR_T_REL_TRANSFORM]) {
    const float gsr = c.gs[GLAMR_T_REL_TRANSFORM];
    const float twt = pb.rel_trans_weight;
    const int i = p;
    for (int j = 0; j < pb.P; ++j) {
      if (j == i) continue;
      const size_t nj = (size_t)j * T + t;
      const float w_ij = pb.rel_w[((size_t)i * pb.P + j) * T + t], wt_ij = pb.rel_wt[((size_t)i * pb.P + j) * T + t];
      const float w_ji = pb.rel_w[((size_t)j * pb.P + i) * T + t], wt_ji = pb.rel_wt[((size_t)j * pb.P + i) * T + t];
      if (w_ij == 0.0f && wt_ij == 0.0f && w_ji == 0.0f && wt_ji == 0.0f) continue;
      float Rj[9];
      aa_to_rotmat(c.sc.orient_world + nj * 3, Rj);
      const float* tj = c.sc.trans_world + nj * 3;
      const float dt[3] = {tj[0] - tw[0], tj[1] - tw[1], tj[2] - tw[2]};
      {  // pair (i,j): R_W = Ri^T Rj, t_W = Ri^T (tj - ti); this thread owns its loss value and dL/dT_i
        const float* C = pb.rel_target + (((size_t)i * pb.P + j) * T + t) * 12;
        float RW[9], tW[3], gRW[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, gtW[3];
        mat3_tmul(Rw, Rj, RW);
        mat3_tvec(Rw, dt, tW);
        float sr = 0.0f, st = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            const float d = C[a * 4 + b] - RW[a * 3 + b];
            sr += d * d;
            gRW[a * 3 + b] = -2.0f * gsr * w_ij * d;
          }
          const float d = C[a * 4 + 3] - tW[a];
          st += d * d;
          gtW[a] = -2.0f * gsr * wt_ij * twt * d;
        }
        acc.v[GLAMR_T_REL_TRANSFORM] += (double)(w_ij * sr + wt_ij * twt * st);
        if (gsr != 0.0f) {
          // R_W = Ri^T Rj -> dRi = Rj gRW^T ; t_W = Ri^T dt -> dRi += dt gtW^T, d ti = -Ri gtW
          float t1[9], g[3];
          mat3_mult(Rj, gRW, t1);
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) g_Rw[a * 3 + b] += t1[a * 3 + b] + dt[a] * gtW[b];
          mat3_vec(Rw, gtW, g);
          g_tw[0] -= g[0]; g_tw[1] -= g[1]; g_tw[2] -= g[2];
          any_Rw = true;
        }
      }
      if (gsr != 0.0f && (w_ji != 0.0f || wt_ji != 0.0f)) {
        // pair (j,i): R_W' = Rj^T Ri, t_W' = Rj^T (ti - tj); only dL/dT_i here (thread (j,t) adds the value)
        const float* C = pb.rel_target + (((size_t)j * pb.P + i) * T + t) * 12;
        float RW[9], tW[3], gRW[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, gtW[3];
        const float mdt[3] = {-dt[0], -dt[1], -dt[2]};
        mat3_tmul(Rj, Rw, RW);
        mat3_tvec(Rj, mdt, tW);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
          for (int b = 0; b < 2; ++b) gRW[a * 3 + b] = -2.0f * gsr * w_ji * (C[a * 4 + b] - RW[a * 3 + b]);
          gtW[a] = -2.0f * gsr * wt_ji * twt * (C[a * 4 + 3] - tW[a]);
        }
        float t1[9], g[3];
        mat3_mul(Rj, gRW, t1);   // dRi = Rj gRW'
#pragma unroll
        for (int k = 0; k < 9; ++k) g_Rw[k] += t1[k];
        mat3_vec(Rj, gtW, g);    // d ti = Rj gtW'
        g_tw[0] += g[0]; g_tw[1] += g[1]; g_tw[2] += g[2];
        any_Rw = true;
      }
    }
  }
  GLAMR_STAMP(8);
  if (any_Rw) {
    float g[3];
    aa_to_rotmat_vjp(ow, g_Rw, g);
    g_ow[0] += g[0]; g_ow[1] += g[1]; g_ow[2] += g[2];
  }
  GLAMR_STAMP(9);
#pragma unroll
  for (int k = 0; k < 3; ++k) { c.sc.g_orient[n * 3 + k] = g_ow[k]; c.sc.g_trans[n * 3 + k] = g_tw[k]; }
#pragma unroll
  for (int k = 0; k < 9; ++k) c.sc.g_cam[n * 12 + k] = g_Rc[k];
#pragma unroll
  for (int k = 0; k < 3; ++k) c.sc.g_cam[n * 12 + 9 + k] = g_tc[k];
}

// Sequential form (host harness): all joints of (p,t), then the rest.
GLAMR_HD void frame_residuals(const OptCtx& c, int p, int t, TermAcc& acc) {
  const size_t n = (size_t)p * c.pb.T + t;
  float Rc[9], tc[3], Rs[9];
  mat34_R(c.sc.cam + (size_t)t * 12, Rc);
  tc[0] = c.sc.cam[(size_t)t * 12 + 3]; tc[1] = c.sc.cam[(size_t)t * 12 + 7]; tc[2] = c.sc.cam[(size_t)t * 12 + 11];
  rodrigues_smplx(c.sc.orient_world + n * 3, Rs);
  KpGrad kg;
  kg.clear();
  for (int k = 0; k < c.pb.J; ++k)
    kp_joint_terms(c, p, t, k, c.sc.joints_world + (n * c.pb.J + k) * 3, Rc, tc, Rs, c.sc.trans_world + n * 3, kg);
  frame_rest(c, p, t, kg, acc);
}

// ------------------------------------------------------------------------------------------------ camera backward
// Per frame t: sum dL/dcam over this rank's persons, add the camera-only terms (loss_func.py:60-114,199-201,240)
// and push the gradient into the camera variables (or, mode 3, into the residual variables and back into the
// persons' world transforms).
GLAMR_HD void camera_backward(const OptCtx& c, int t, TermAcc& acc) {
  const glamr_problem_t& pb = c.pb;
  const int T = pb.T;
  float G[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // dL/dRc (9) , dL/dtc (3)
  for (int p = 0; p < pb.P; ++p) {          // frame-persons of other ranks hold zeros (frame_residuals_kernel)
    const float* g = c.sc.g_cam + ((size_t)p * T + t) * 12;
#pragma unroll
    for (int k = 0; k < 12; ++k) G[k] += g[k];
  }
  const float* cam = c.sc.cam + (size_t)t * 12;
  const float* inv = c.sc.cam_inv + (size_t)t * 12;
  float gRi[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, gti[3] = {0, 0, 0};   // w.r.t. cam_inv
  if (pb.owner) {
    if (pb.term_enabled[GLAMR_T_CAM_INV_ROT_SMOOTH] && T > 1) {
      const float gs = c.gs[GLAMR_T_CAM_INV_ROT_SMOOTH];
      float ss = 0.0f;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          const float x = inv[a * 4 + b];
          if (t + 1 < T) { const float d = x - inv[12 + a * 4 + b]; ss += d * d; gRi[a * 3 + b] += 2.0f * kFps2 * gs * d; }
          if (t > 0) gRi[a * 3 + b] -= 2.0f * kFps2 * gs * (inv[-12 + a * 4 + b] - x);
        }
      acc.v[GLAMR_T_CAM_INV_ROT_SMOOTH] += (double)(kFps2 * ss);
    }
    if (pb.term_enabled[GLAMR_T_CAM_ORIGIN_SMOOTH] && T > 1) {
      const float gs = c.gs[GLAMR_T_CAM_ORIGIN_SMOOTH];
      float ss = 0.0f;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float x = inv[a * 4 + 3];
        if (t + 1 < T) { const float d = inv[12 + a * 4 + 3] - x; ss += d * d; gti[a] -= 2.0f * kFps2 * gs * d; }
        if (t > 0) gti[a] += 2.0f * kFps2 * gs * (x - inv[-12 + a * 4 + 3]);
      }
      acc.v[GLAMR_T_CAM_ORIGIN_SMOOTH] += (double)(kFps2 * ss);
    }
    if (pb.term_enabled[GLAMR_T_CAM_DEPTH_SMOOTH] && T > 1) {
      // loss_func.py:94-103: velocity of the camera origin along the NEXT frame's optical axis (third column of
      // cam_pose_inv[t+1]), squared and SUMMED over the T-1 frame pairs (the trailing .mean() acts on a 0-d tensor)
      const float gs = c.gs[GLAMR_T_CAM_DEPTH_SMOOTH];
      if (t + 1 < T) {            // pair (t, t+1): this frame is the "previous" origin
        float d = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) d += (inv[a * 4 + 3] - inv[12 + a * 4 + 3]) * inv[12 + a * 4 + 2];
#pragma unroll
        for (int a = 0; a < 3; ++a) gti[a] += 2.0f * kFps2 * gs * d * inv[12 + a * 4 + 2];
        acc.v[GLAMR_T_CAM_DEPTH_SMOOTH] += (double)(kFps2 * d * d);
      }
      if (t > 0) {                // pair (t-1, t): this frame supplies the origin that is subtracted and the axis
        float d = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) d += (inv[-12 + a * 4 + 3] - inv[a * 4 + 3]) * inv[a * 4 + 2];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          gti[a] -= 2.0f * kFps2 * gs * d * inv[a * 4 + 2];
          gRi[a * 3 + 2] += 2.0f * kFps2 * gs * d * (inv[-12 + a * 4 + 3] - inv[a * 4 + 3]);
        }
      }
    }
    if (pb.term_enabled[GLAMR_T_CAM_UP_REG]) {
      float w = (t < 10) ? pb.cam_up_first_weight : 1.0f;
      if (pb.cam_up_first_only && t > 0) w = 0.0f;
      acc.v[GLAMR_T_CAM_UP_REG] += (double)(w * inv[2 * 4 + 1]);
      gRi[2 * 3 + 1] += c.gs[GLAMR_T_CAM_UP_REG] * w;
    }
  }
  const int mode = pb.cam_mode;
  if (mode == GLAMR_CAM_PER_FRAME || mode == GLAMR_CAM_FIXED) {
    // cam_inv = [Rc^T | -Rc^T tc]:  dRc += gRi^T - tc gti^T ,  dtc += -Rc gti
    float Rc[9];
    mat34_R(cam, Rc);
    const float tc[3] = {cam[3], cam[7], cam[11]};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) G[a * 3 + b] += gRi[b * 3 + a] - tc[a] * gti[b];
    float r[3];
    mat3_vec(Rc, gti, r);
    G[9] -= r[0]; G[10] -= r[1]; G[11] -= r[2];
    const int row = (mode == GLAMR_CAM_FIXED) ? 0 : t;
    float g6[6];
    rot6d_to_rotmat_vjp(c.theta + pb.off_cam_rot + 6 * row, G, g6);
    float gtr[3] = {G[9], G[10], G[11]};
    if (pb.owner && mode == GLAMR_CAM_PER_FRAME) {
      // smoothness directly on the camera variables (loss_func.py:60-73)
      if (pb.term_enabled[GLAMR_T_CAM_ROT_SMOOTH] && T > 1) {
        const float gs = c.gs[GLAMR_T_CAM_ROT_SMOOTH];
        const float* x = c.theta + pb.off_cam_rot + 6 * t;
        float ss = 0.0f;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          if (t + 1 < T) { const float d = x[k] - x[6 + k]; ss += d * d; g6[k] += 2.0f * kFps2 * gs * d; }
          if (t > 0) g6[k] -= 2.0f * kFps2 * gs * (x[k - 6] - x[k]);
        }
        acc.v[GLAMR_T_CAM_ROT_SMOOTH] += (double)(kFps2 * ss);
      }
      if (pb.term_enabled[GLAMR_T_CAM_TRANS_SMOOTH] && T > 1) {
        const float gs = c.gs[GLAMR_T_CAM_TRANS_SMOOTH];
        const float* x = c.theta + pb.off_cam_trans + 3 * t;
        float ss = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          if (t + 1 < T) { const float d = x[k] - x[3 + k]; ss += d * d; gtr[k] += 2.0f * kFps2 * gs * d; }
          if (t > 0) gtr[k] -= 2.0f * kFps2 * gs * (x[k - 3] - x[k]);
        }
        acc.v[GLAMR_T_CAM_TRANS_SMOOTH] += (double)(kFps2 * ss);
      }
    }
    if (mode == GLAMR_CAM_PER_FRAME) {
#pragma unroll
      for (int k = 0; k < 6; ++k) c.sc.grad[pb.off_cam_rot + 6 * t + k] = g6[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) c.sc.grad[pb.off_cam_trans + 3 * t + k] = gtr[k];
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) c.sc.g_cam_fix[(size_t)t * 12 + k] = g6[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) c.sc.g_cam_fix[(size_t)t * 12 + 6 + k] = gtr[k];
    }
  } else if (mode == GLAMR_CAM_FROM_PERSONS) {
    // cam = inverse(cam_inv): Rc = Ri^T, tc = -Ri^T ti  ->  dRi += G_R^T - ti G_t^T ,  dti += -Ri G_t
    float Ri[9];
    mat34_R(inv, Ri);
    const float ti[3] = {inv[3], inv[7], inv[11]};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) gRi[a * 3 + b] += G[b * 3 + a] - ti[a] * G[9 + b];
    float r[3];
    const float Gt[3] = {G[9], G[10], G[11]};
    mat3_vec(Ri, Gt, r);
    gti[0] -= r[0]; gti[1] -= r[1]; gti[2] -= r[2];
    float g6[6];
    rot6d_to_rotmat_vjp(c.sc.cam_d6 + (size_t)t * 6, gRi, g6);
    const int e = pb.empty_index[t];
    if (e >= 0) {
#pragma unroll
      for (int k = 0; k < 6; ++k) c.sc.grad[pb.off_cam_rot + 6 * e + k] = g6[k];
    }
    // cam_inv_trans_residual_reg (loss_func.py:199-201,:240): sum (30 x)^2 / rows, owner only
    const int trow = pb.trans_res_all ? t : e;
    if (trow >= 0) {
      float gr[3] = {gti[0], gti[1], gti[2]};
      if (pb.owner && pb.term_enabled[GLAMR_T_CAM_INV_TRANS_RES_REG]) {
        const float gs = c.gs[GLAMR_T_CAM_INV_TRANS_RES_REG];
        float ss = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) { const float x = c.theta[pb.off_cam_trans + 3 * trow + k]; ss += x * x; gr[k] += 2.0f * kFps2 * gs * x; }
        acc.v[GLAMR_T_CAM_INV_TRANS_RES_REG] += (double)(kFps2 * ss);
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) c.sc.grad[pb.off_cam_trans + 3 * trow + k] = gr[k];
    }
    // stash dL/d(mean cam_inv) of this frame in g_cam_fix for the scatter to the source frame
    float gR[9];
    rotmat_to_rot6d_vjp(g6, gR);
#pragma unroll
    for (int k = 0; k < 9; ++k) c.sc.g_cam_fix[(size_t)t * 12 + k] = gR[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) c.sc.g_cam_fix[(size_t)t * 12 + 9 + k] = gti[k];
  }
}
// mode 3 only, after camera_backward of all frames: frame s gathers dL/d(mean) of every frame filled from it and
// pushes it into dL/d(person_transform_world) of its visible persons (and into their person2cam residuals, if any).
GLAMR_HD void camera_scatter_to_persons(const OptCtx& c, int s) {
  const glamr_problem_t& pb = c.pb;
  const int T = pb.T;
  if (pb.fill_src[s] != s || pb.inv_num_persons[s] == 0.0f) return;
  float G[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int t = 0; t < T; ++t) {
    if (pb.fill_src[t] != s) continue;
    const float* g = c.sc.g_cam_fix + (size_t)t * 12;
#pragma unroll
    for (int k = 0; k < 12; ++k) G[k] += g[k];
  }
  const float inv_n = pb.inv_num_persons[s];
#pragma unroll
  for (int k = 0; k < 12; ++k) G[k] *= inv_n;
  for (int p = 0; p < pb.P; ++p) {
    const glamr_person_t& ps = pb.persons[p];
    if (ps.vis[s] == 0.0f) continue;
    // M = Tw @ P2C: R_M = Rw Rp, t_M = Rw tp + tw  ->  dRw = G_R Rp^T + G_t tp^T, dtw = G_t
    float P2Cbuf[12], Rp[9], gRw[9], g[3];
    const float* P2C = person2cam_at(c, ps, s, P2Cbuf);
    mat34_R(P2C, Rp);
    mat3_mult(G, Rp, gRw);
    const float tp[3] = {P2C[3], P2C[7], P2C[11]};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) gRw[a * 3 + b] += G[9 + a] * tp[b];
    const size_t n = (size_t)p * T + s;
    aa_to_rotmat_vjp(c.sc.orient_world + n * 3, gRw, g);
#pragma unroll
    for (int k = 0; k < 3; ++k) { c.sc.g_orient[n * 3 + k] += g[k]; c.sc.g_trans[n * 3 + k] += G[9 + k]; }
    const int o = ps.off_person2cam_res;
    if (o >= 0) {
      // P2C = P2C0 @ [Rr | tr]: R_M = Rw R0 Rr, t_M = Rw (R0 tr + t0) + tw  ->  dRr = (Rw R0)^T G_R, dtr = (Rw R0)^T G_t.
      // Linear in G like the lines above: with several ranks each writes its share and the all-reduce adds them.
      float Rw[9], R0[9], A[9], gRr[9], g6[6], gtr[3];
      aa_to_rotmat(c.sc.orient_world + n * 3, Rw);
      mat34_R(ps.person2cam + (size_t)s * 12, R0);
      mat3_mul(Rw, R0, A);
      mat3_tmul(A, G, gRr);
      mat3_tvec(A, G + 9, gtr);
      rot6d_to_rotmat_vjp(c.theta + o + 6 * s, gRr, g6);
#pragma unroll
      for (int k = 0; k < 6; ++k) c.sc.grad[o + 6 * s + k] = g6[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) c.sc.grad[o + 6 * T + 3 * s + k] = gtr[k];
    }
  }
}

// ------------------------------------------------------------------------------------------------ trajectory bwd
// Reverse of traj_post for absolute frame t: world compose -> base pose -> quaternion chain.  Writes the gradients
// of world_dheading / world_res / local_rot / local_z, and seeds the two reverse scans (g_xy, g_head).
GLAMR_HD void traj_back_pre(const OptCtx& c, int p, int t, TermAcc& acc) {
  const glamr_problem_t& pb = c.pb;
  const glamr_person_t& ps = pb.persons[p];
  const int T = pb.T;
  const size_t n = (size_t)p * T + t;
  const int i = t - ps.start;
  float g_ow[3], g_tw[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { g_ow[k] = c.sc.g_orient[n * 3 + k]; g_tw[k] = c.sc.g_trans[n * 3 + k]; }
  const float* ob = c.sc.orient_base + n * 3;
  float g_ob[3] = {g_ow[0], g_ow[1], g_ow[2]}, g_tb[3] = {g_tw[0], g_tw[1], g_tw[2]};
  if (pb.use_world_res) {
    // traj_rot_res / traj_trans_res regularisers (loss_func.py:204-209) on the owner rank
    float go[3] = {g_ow[0], g_ow[1], g_ow[2]}, gt[3] = {g_tw[0], g_tw[1], g_tw[2]};
    if (pb.owner) {
      if (pb.term_enabled[GLAMR_T_ROT_RES]) {
        float ss = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) { const float x = c.theta[ps.off_orient_res + t * 3 + k]; ss += x * x; go[k] += 2.0f * kFps2 * c.gs[GLAMR_T_ROT_RES] * x; }
        acc.v[GLAMR_T_ROT_RES] += (double)(kFps2 * ss);
      }
      if (pb.term_enabled[GLAMR_T_TRANS_RES]) {
        float ss = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) { const float x = c.theta[ps.off_trans_res + t * 3 + k]; ss += x * x; gt[k] += 2.0f * kFps2 * c.gs[GLAMR_T_TRANS_RES] * x; }
        acc.v[GLAMR_T_TRANS_RES] += (double)(kFps2 * ss);
      }
    }
    if (!pb.has_world_dheading) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { c.sc.grad[ps.off_orient_res + t * 3 + k] = go[k]; c.sc.grad[ps.off_trans_res + t * 3 + k] = gt[k]; }
    } else {
      // world_dheading overrides the residual branch (:459-465): residuals get only their regulariser gradient
#pragma unroll
      for (int k = 0; k < 3; ++k) { c.sc.grad[ps.off_orient_res + t * 3 + k] = go[k] - g_ow[k]; c.sc.grad[ps.off_trans_res + t * 3 + k] = gt[k] - g_tw[k]; }
    }
  }
  if (pb.has_world_dheading) {
    const float da[3] = {0.0f, 0.0f, c.theta[ps.off_world_dheading + t]};
    float dq[4], bq[4], q[4], gq[4], gdq[4], gbq[4], gda[3];
    aa_to_quat(da, dq);
    aa_to_quat(ob, bq);
    quat_mul(dq, bq, q);
    quat_to_aa_vjp(q, g_ow, gq);
    quat_mul_vjp(dq, bq, gq, gdq, gbq);
    aa_to_quat_vjp(da, gdq, gda);
    c.sc.grad[ps.off_world_dheading + t] = gda[2];
    aa_to_quat_vjp(ob, gbq, g_ob);
  }
  float g_heading = 0.0f, g_x = 0.0f, g_y = 0.0f;
  if (i >= 0 && i < ps.len) {
    const float* tl = c.sc.traj_local + n * 11;
    float q_hl[4], lq[4], hq[4], q[4], gq[4], gq_hl[4], ghq[4], glq[4];
    local_quat(tl + 3, c.sc.heading[n], q_hl, lq, hq);
    const float base[4] = {0.5f, 0.5f, 0.5f, 0.5f};
    quat_mul(q_hl, base, q);
    quat_to_aa_vjp(q, g_ob, gq);
    quat_mul_vjp(q_hl, base, gq, gq_hl, nullptr);
    quat_mul_vjp(hq, lq, gq_hl, ghq, glq);
    const float ha[3] = {0.0f, 0.0f, c.sc.heading[n]};
    float gha[3];
    aa_to_quat_vjp(ha, ghq, gha);
    g_heading = gha[2];
    float R[9], gR[9], g6[6];
    rot6d_to_rotmat(tl + 3, R);
    rotmat_to_quat_vjp(R, glq, gR);
    rot6d_to_rotmat_vjp(tl + 3, gR, g6);
    const float rm = ps.rot_mask ? ps.rot_mask[i] : 1.0f;
    float ssr = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float x = c.theta[ps.off_rot + 6 * i + k];
      float g = g6[k] * rm;
      if (pb.owner) { ssr += x * x; g += 2.0f * kFps2 * c.gs[GLAMR_T_ROT_REG] * x; }
      c.sc.grad[ps.off_rot + 6 * i + k] = g;
    }
    {
      const float x = c.theta[ps.off_z + i];
      float g = g_tb[2];
      if (pb.owner) {
        g += 2.0f * kFps2 * c.gs[GLAMR_T_Z_REG] * x;
        if (pb.term_enabled[GLAMR_T_Z_REG]) acc.v[GLAMR_T_Z_REG] += (double)(kFps2 * x * x);
        if (pb.term_enabled[GLAMR_T_ROT_REG]) acc.v[GLAMR_T_ROT_REG] += (double)(kFps2 * ssr);
      }
      c.sc.grad[ps.off_z + i] = g;
    }
    g_x = g_tb[0];
    g_y = g_tb[1];
  }
  c.sc.g_xy[2 * n] = g_x;
  c.sc.g_xy[2 * n + 1] = g_y;
  c.sc.g_head[n] = g_heading;
}
// after the reverse inclusive scan of g_xy over the local frames: rot_2d backward (traj_utils.py:7-11,:76)
GLAMR_HD void traj_back_mid(const OptCtx& c, int p, int i, TermAcc& acc) {
  const glamr_problem_t& pb = c.pb;
  const glamr_person_t& ps = pb.persons[p];
  const size_t n = (size_t)p * pb.T + ps.start + i;
  const float Gx = c.sc.g_xy[2 * n], Gy = c.sc.g_xy[2 * n + 1];
  if (i == 0) {
    c.sc.grad[ps.off_xy] = Gx;
    c.sc.grad[ps.off_xy + 1] = Gy;
  } else {
    const float t = c.sc.heading[n - 1];
    const float ct = cosf(t), st = sinf(t);
    float gx = Gx * ct + Gy * st, gy = -Gx * st + Gy * ct;
    const float x = c.theta[ps.off_dxy + 2 * (i - 1)], y = c.theta[ps.off_dxy + 2 * (i - 1) + 1];
    if (pb.owner) {
      gx += 2.0f * kFps2 * c.gs[GLAMR_T_DXY_REG] * x;
      gy += 2.0f * kFps2 * c.gs[GLAMR_T_DXY_REG] * y;
      if (pb.term_enabled[GLAMR_T_DXY_REG]) acc.v[GLAMR_T_DXY_REG] += (double)(kFps2 * (x * x + y * y));
    }
    c.sc.grad[ps.off_dxy + 2 * (i - 1)] = gx;
    c.sc.grad[ps.off_dxy + 2 * (i - 1) + 1] = gy;
  }
  // heading[i] rotates d_xy of frame i+1: add that dependence to this frame's own heading gradient
  if (i + 1 < ps.len) {
    const float* tl = c.sc.traj_local + (n + 1) * 11;
    const float Gx1 = c.sc.g_xy[2 * (n + 1)], Gy1 = c.sc.g_xy[2 * (n + 1) + 1];
    const float t = c.sc.heading[n];
    const float ct = cosf(t), st = sinf(t);
    c.sc.g_head[n] += Gx1 * (-tl[0] * st - tl[1] * ct) + Gy1 * (tl[0] * ct - tl[1] * st);
  }
}
// after the reverse inclusive scan of g_head: heading variables + dheading regularisers (loss_func.py:216-230)
GLAMR_HD void traj_back_post(const OptCtx& c, int p, int i, TermAcc& acc) {
  const glamr_problem_t& pb = c.pb;
  const glamr_person_t& ps = pb.persons[p];
  const size_t n = (size_t)p * pb.T + ps.start + i;
  const float G = c.sc.g_head[n];
  if (i == 0) {
    c.sc.grad[ps.off_heading] = G;
  } else {
    const float x = c.theta[ps.off_dheading + i - 1];
    float g = G * ps.dheading_mask[i - 1];
    if (pb.owner) {
      const float sx = sinf(x), cx = cosf(x);
      g += 2.0f * kFps2 * c.gs[GLAMR_T_DHEADING_REG] * x + 2.0f * kFps2 * c.gs[GLAMR_T_DHEADING_REG_NEW] * sx;
      if (pb.term_enabled[GLAMR_T_DHEADING_REG]) acc.v[GLAMR_T_DHEADING_REG] += (double)(kFps2 * x * x);
      if (pb.term_enabled[GLAMR_T_DHEADING_REG_NEW]) acc.v[GLAMR_T_DHEADING_REG_NEW] += (double)(kFps2 * ((cx - 1.0f) * (cx - 1.0f) + sx * sx));
    }
    c.sc.grad[ps.off_dheading + i - 1] = g;
  }
}

// torch.optim.Adam (betas 0.9/0.999, eps 1e-8, no weight decay, no amsgrad); `step` is 1-based
GLAMR_HD void adam_update(float& p, float g, float& m, float& v, float lr, float bc1, float bc2_sqrt) {
  m = m + 0.1f * (g - m);                     // exp_avg.lerp_(grad, 1 - beta1)
  v = 0.999f * v + 0.001f * g * g;
  const float denom = sqrtf(v) / bc2_sqrt + 1e-8f;
  p -= (lr / bc1) * (m / denom);
}

}  // namespace glamr
