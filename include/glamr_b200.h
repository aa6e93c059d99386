/* glamr_b200 -- C ABI of the B200 (sm_100a) CUDA library behind GLAMR's global-reconstruction path.
 *
 * GLAMR (NVlabs/GLAMR) is pure Python/PyTorch: it has no FFI layer, the seams a replacement binds to are Python
 * call sites.  Each entry point below names the reference interface it stands behind (paths relative to the
 * reference tree).  The Python host code in glamr_b200/ binds these with ctypes (INTEGRATION.md shows the stub a
 * GLAMR maintainer would add).
 *
 * Conventions: plain C, no torch types.  Unless stated otherwise every pointer is a DEVICE pointer to contiguous
 * row-major float32; `stream` is a cudaStream_t passed as void*.  Functions return 0 on success, a cudaError_t
 * value (>0) for CUDA failures, or a negative GLAMR_E* code for argument errors.  They never synchronise the
 * stream and never allocate device memory, except the *_create functions whose allocations are owned by the
 * returned opaque handle and released by *_destroy.  All buffers are caller-owned.  Re-entrant across streams; no
 * global state.
 */
#ifndef GLAMR_B200_H
#define GLAMR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLAMR_OK 0
#define GLAMR_EINVAL (-1)      /* bad argument / unsupported shape */
#define GLAMR_ENOSPACE (-2)    /* workspace too small */
#define GLAMR_EUNSUPPORTED (-3)

#define GLAMR_NUM_VERTS 6890
#define GLAMR_NUM_JOINTS 24
#define GLAMR_NUM_BETAS 10
#define GLAMR_NUM_POSE_FEAT 207

int glamr_version(void);
/* number of SMs / device ordinal the library sees for the current context (for grid sizing diagnostics) */
int glamr_device_sm_count(void);
/* Measurement aid: launches a register-resident FFMA loop (8 CTAs x 256 threads per SM, 16 independent chains, `iters`
 * rounds) on `stream`; *flops (HOST pointer) receives the flop count of the launch.  The caller times it with events: the
 * FP32 throughput this GPU sustains at its present clocks (bench.py's roofline.fp32.peak).  scratch: >= 8*256*SMs floats. */
int glamr_fp32_probe(int iters, float* scratch, size_t scratch_floats, double* flops, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * SMPL body model  --  stands behind lib/models/smpl.py:274-343 (class SMPL: forward, get_joints) and the
 * third-party smplx.lbs it calls (in-tree statement: HybrIK/hybrik/models/layers/smpl/lbs.py:195-288,402-548).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct glamr_smpl glamr_smpl_t;

/* All constant arrays are HOST pointers (one-off upload; the library re-tiles them for its kernels).
 *   v_template [6890,3]  shapedirs [6890,3,10]  posedirs [207,20670]  J_regressor [24,6890]
 *   lbs_weights [6890,24]  parents [24]  J_regressor_extra [n_extra,6890]
 *   pick_vertex_ids [n_picks]  (smplx VertexJointSelector)     joint_map [n_map] indexes [24 | n_picks | n_extra]
 */
int glamr_smpl_create(glamr_smpl_t** out, const float* v_template, const float* shapedirs, const float* posedirs,
                      const float* J_regressor, const float* lbs_weights, const int32_t* parents,
                      const float* J_regressor_extra, int n_extra, const int32_t* pick_vertex_ids, int n_picks,
                      const int32_t* joint_map, int n_map);
int glamr_smpl_destroy(glamr_smpl_t* m);
/* introspection: 0 max skin weights per vertex, 1 support size (vertices feeding picks/regressors), 2 n_map */
int glamr_smpl_info(const glamr_smpl_t* m, int what);
size_t glamr_smpl_workspace_bytes(const glamr_smpl_t* m, int n);       /* glamr_smpl_forward */
size_t glamr_smpl_fk_workspace_bytes(const glamr_smpl_t* m, int n);    /* glamr_smpl_fk24 (no blend operands) */
/* Which kernels evaluate the blend + skinning of SMPL.forward: 1 (default) = tcgen05 3xTF32 blend GEMM + skinning kernel,
 * 0 = the single FP32 SIMT kernel (kept for A/B verification; env GLAMR_LBS_PATH=simt selects it at start-up).  Process-wide. */
int glamr_smpl_set_lbs_path(int path);

/* SMPL.forward (lib/models/smpl.py:289-316).  n frame-persons.
 *   global_orient [n,3] (NULL -> zeros)  body_pose [n,69]  betas [n,10]
 *   root_trans [n,3] or NULL (no re-rooting)   root_scale [n] or NULL (-> 1)
 *   orig_joints != 0: joints = the 24 LBS joints, else the n_map mapped joints
 *   joints [n, 24 or n_map, 3]   vertices [n,6890,3] or NULL
 */
int glamr_smpl_forward(const glamr_smpl_t* m, int n, const float* global_orient, const float* body_pose,
                       const float* betas, const float* root_trans, const float* root_scale, int orig_joints,
                       float* joints, float* vertices, void* workspace, size_t workspace_bytes, void* stream);

/* SMPL.get_joints (lib/models/smpl.py:318-343): FK only, rest joints from v_template (betas ignored). */
int glamr_smpl_fk24(const glamr_smpl_t* m, int n, const float* global_orient, const float* body_pose,
                    const float* root_trans, const float* root_scale, float* joints, void* workspace,
                    size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Row-wise rotation algebra  --  lib/utils/konia_transform.py:234-822, lib/utils/torch_transform.py:10-279.
 * op codes: see glamr_b200/csrc/rowops.cuh (RowOp).  in1 may be NULL for unary ops; gin* may be NULL.
 * ---------------------------------------------------------------------------------------------------------- */
int glamr_rowop_fwd(int op, int n, const float* in0, const float* in1, float* out, void* stream);
int glamr_rowop_vjp(int op, int n, const float* in0, const float* in1, const float* gout, float* gin0,
                    float* gin1, void* stream);

/* traj_pred/utils/traj_utils.py:65-88  traj_local2global_heading for B sequences of T frames, time-major
 * local_traj [T,B,11] -> trans [T,B,3], orient_q [T,B,4] (local_orient_type '6d', local_heading on/off);
 * scratch [B*T*3] floats */
int glamr_traj_local2global(int T, int B, const float* local_traj, int local_heading, float* trans, float* orient_q,
                            float* scratch, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Learned prior (inference only)  --  stands behind MotionTrajJointModel.inference
 * (motion_infiller/models/motion_traj_joint_model.py:141-145): MotionInfillerVAE.inference_one_step
 * (motion_infiller/models/motion_infiller_vae.py:551-562 with ContextEncoder :92-123, DataDecoder :345-421) and
 * TrajPredVAE.inference (traj_pred/models/traj_pred_vae.py:524-548 with ContextEncoder :72-92, DataDecoder :269-333).
 * Parameters are registered under their reference state-dict names ("context_encoder.in_fc.weight", ...), so a
 * Lightning checkpoint's state_dict maps 1:1.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct glamr_net glamr_net_t;
int glamr_net_create(glamr_net_t** out);
int glamr_net_destroy(glamr_net_t* n);
/* upload one named float32 parameter from a HOST pointer */
int glamr_net_set_tensor(glamr_net_t* n, const char* name, const float* host, size_t numel);
/* Y[M,N] = act(X[M,K] W[N,K]^T + bias): the GEMM behind every nn.Linear / attention projection / FFN of the prior
 * networks.  mode 1 (default inside the networks): tcgen05.mma.kind::tf32 with a 3xTF32 split (FP32-accurate), TMEM
 * accumulator; mode 0: FP32 SIMT kernel kept for A/B verification.  bias may be NULL. */
int glamr_linear_forward(int M, int N, int K, const float* X, const float* W, const float* bias, int relu, float* Y, int mode,
                         void* stream);
int glamr_net_set_gemm_mode(int mode);
size_t glamr_infiller_workspace_floats(int B);
size_t glamr_trajpred_workspace_floats(int T, int B);
/* One 50-frame window (past 10 | current 30 | future 10), B sequences, seq-first buffers:
 *   in_pose [50,B,69]   key_pad_mask [B,50] uint8 (1 = frame invisible / padding)   eps [eps_rows,128], eps_rows in {1,B}, or NULL
 *   out_pose [40,B,69] = the 10 past input frames followed by the 30 decoded frames */
int glamr_infiller_window_forward(const glamr_net_t* n, int B, const float* in_pose, const uint8_t* key_pad_mask,
                                  const float* eps, int eps_rows, float* out_pose, float* workspace, size_t workspace_floats,
                                  void* stream);
/* The whole autoregressive sweep of motion_infiller_vae.py:618-632 (windows of 50 frames, stride 30) in one call:
 *   pose_io [T,B,69]: input body pose, overwritten with the infilled pose   key_pad_all [B,T] uint8 (1 = frame invisible)
 *   eps [ceil((T-10)/30)][eps_rows][128], eps_rows in {1,B}   workspace >= glamr_infiller_sequence_workspace_floats(B) floats */
size_t glamr_infiller_sequence_workspace_floats(int B);
int glamr_infiller_forward(const glamr_net_t* n, int T, int B, float* pose_io, const uint8_t* key_pad_all, const float* eps,
                           int eps_rows, float* workspace, size_t workspace_floats, void* stream);
/*   in_joint_pos [T,B,69] (23 joints from SMPL.get_joints)   eps as above   init_xy [B,2] / init_heading [B] or NULL
 *   out_local_traj [T,B,11]   out_trans [T,B,3]   out_orient_aa [T,B,3] */
int glamr_trajpred_forward(const glamr_net_t* n, int T, int B, const float* in_joint_pos, const float* eps, int eps_rows,
                           const float* init_xy, const float* init_heading, float* out_local_traj, float* out_trans,
                           float* out_orient_aa, float* workspace, size_t workspace_floats, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Global optimisation  --  stands behind GlobalReconOptimizer.forward / compute_loss / optimize_main
 * (global_recon/models/global_recon_model.py:428-570), the residual registry global_recon/models/loss_func.py:314-340
 * and torch.optim.Adam.step (:563,:642).
 * ---------------------------------------------------------------------------------------------------------- */
enum glamr_term {
  GLAMR_T_KP_2D = 0, GLAMR_T_KP_2D_DIST, GLAMR_T_CAM_TRAJ_ROT, GLAMR_T_CAM_TRAJ_TRANS, GLAMR_T_TRAJ_ROT_SMOOTH,
  GLAMR_T_TRAJ_TRANS_SMOOTH, GLAMR_T_REL_TRANSFORM, GLAMR_T_DXY_REG, GLAMR_T_DHEADING_REG, GLAMR_T_DHEADING_REG_NEW,
  GLAMR_T_ROT_REG, GLAMR_T_Z_REG, GLAMR_T_ROT_RES, GLAMR_T_TRANS_RES, GLAMR_T_CAM_INV_TRANS_RES_REG,
  GLAMR_T_CAM_INV_ROT_SMOOTH, GLAMR_T_CAM_ORIGIN_SMOOTH, GLAMR_T_CAM_UP_REG, GLAMR_T_CAM_ROT_SMOOTH,
  GLAMR_T_CAM_TRANS_SMOOTH, GLAMR_T_CAM_DEPTH_SMOOTH, GLAMR_NUM_TERMS
};

enum glamr_cam_mode {
  GLAMR_CAM_CONST = 0,        /* camera is data (cam_pose_const)                           (:473 not taken)      */
  GLAMR_CAM_PER_FRAME = 1,    /* variables cam_rot_6d [T,6], cam_trans [T,3]               (:478-480)            */
  GLAMR_CAM_FIXED = 2,        /* variables cam_rot_6d_fix [1,6], cam_trans_fix [1,3]       (:475-477)            */
  GLAMR_CAM_FROM_PERSONS = 3  /* mean of person_transform_world @ person2cam + residuals   (:481-508)            */
};

typedef struct glamr_person {
  int32_t start, len;              /* exist range [start, start+len) of this person (exist_frames)              */
  int32_t off_xy, off_heading, off_dxy, off_dheading, off_z, off_rot;     /* offsets into theta (floats)        */
  int32_t off_world_dheading, off_orient_res, off_trans_res;              /* [T], [T,3], [T,3]                  */
  int32_t off_person2cam_res;      /* person2cam_res_rot [T,6] followed directly by person2cam_res_trans [T,3], or -1
                                    * (flag_opt_person2cam_* off).  GLAMR_CAM_FROM_PERSONS composes
                                    * person2cam @ [R(rot6d) | trans] (global_recon_model.py:484-488)           */
  const float* traj_local_pred;    /* [len,11]                                                                    */
  const float* orient_base_init;   /* [T,3] smpl_orient_world_base outside the exist range                        */
  const float* trans_base_init;    /* [T,3]                                                                       */
  const float* cam_K;              /* [T,9]                                                                       */
  const float* kp_target;          /* [T,J,2] kp_2d_aligned                                                       */
  const float* orient_cam_6d;      /* [T,6]  rot6d(R(smpl_orient_cam)), target of cam_traj_rot                    */
  const float* orient_cam_q;       /* [T,4]  angle_axis_to_quaternion(smpl_orient_cam): target when rot_type 'quat' */
  const float* trans_cam;          /* [T,3]  root_trans_cam                                                       */
  const float* person2cam;         /* [T,12] 3x4, used by GLAMR_CAM_FROM_PERSONS (before the residual above)      */
  const float* dheading_mask;      /* [len-1] (cam_fix_frames)                                                    */
  const float* rot_mask;           /* [len] or NULL (flag_opt_vis_local_rot)                                      */
  const float* vis;                /* [T] 1/0 vis_frames                                                          */
  /* per-stage weights, already containing score^2, min_conf, first-frame weighting, visibility               */
  const float* kp_w;               /* [T,J]                                                                       */
  const float* kp_dist_mask;       /* [T,J]                                                                       */
  const float* ctr_w;              /* [T]  cam_traj_rot                                                           */
  const float* ctt_w;              /* [T]  cam_traj_trans                                                         */
} glamr_person_t;

typedef struct glamr_problem {
  int32_t P, T, J;                 /* persons, frames, joints per person (n_map of the SMPL handle)              */
  int32_t cam_mode;                /* enum glamr_cam_mode                                                         */
  int32_t off_cam_rot, off_cam_trans; /* variable offsets (modes 1,2: cam_rot_6d / cam_trans; mode 3: residuals)  */
  int32_t use_world_res, has_world_dheading;
  int32_t trans_res_all;           /* mode 3: cam_inv_trans_residual has T rows (else one row per empty frame)    */
  int32_t cam_up_first_only;
  int32_t n_params;                /* length of theta / grad / adam state                                         */
  int32_t n_begin, n_end;          /* frame-persons n = p*T + t whose SMPL / per-frame residuals this rank evaluates
                                    * (multi-GPU shard; any contiguous range, a person may straddle two ranks)         */
  int32_t owner;                   /* != 0: this rank also evaluates the replicated terms (camera, regs, rel)    */
  int32_t cam_traj_rot_quat;       /* cam_traj_rot: rot_type 'quat' (loss_func.py:158-161) instead of '6d'          */
  int32_t traj_rot_smooth_quat;    /* traj_rot_smoothness: rot_type 'quat' (loss_func.py:126-128)                  */
  float cam_up_first_weight;
  float rel_trans_weight;
  float term_weight[GLAMR_NUM_TERMS];   /* YAML weight, 0 if the term is absent                                  */
  float term_norm[GLAMR_NUM_TERMS];     /* normaliser (denominator) of the reference's mean                      */
  int32_t term_enabled[GLAMR_NUM_TERMS];
  int32_t term_monitor[GLAMR_NUM_TERMS];
  const glamr_person_t* persons;   /* DEVICE array [P]                                                            */
  const float* smpl_pose_all;      /* [P,T,69] body pose (infilled), constant during optimisation                 */
  const float* smpl_beta_all;      /* [P,T,10]                                                                    */
  const float* scale_all;          /* [P,T] or NULL                                                               */
  const float* cam_pose_const;     /* [T,12] world->cam 3x4 (mode 0)                                              */
  const int32_t* empty_index;      /* [T] row of cam_inv_rot_residual for frames without any person, else -1     */
  const int32_t* fill_src;         /* [T] forward-fill source frame (mode 3)                                      */
  const float* inv_num_persons;    /* [T] 1/num visible persons (0 where none)                                    */
  const float* rel_target;         /* [P*P,T,12] rel_transform_cam (i*P+j), or NULL                               */
  const float* rel_w;              /* [P*P,T] squared frame weights for the rotation part (0 = frame unused)      */
  const float* rel_wt;             /* [P*P,T] same for the translation part                                       */
  const uint8_t* active;           /* [n_params] 1 where Adam updates theta                                       */
} glamr_problem_t;

size_t glamr_sizeof_person(void);
size_t glamr_sizeof_problem(void);

typedef struct glamr_opt glamr_opt_t;

/* The handle owns scratch sized for (P,T,J) and the Adam moments.  `problem` is copied (host struct; its embedded
 * pointers are device pointers that must stay alive while the handle uses them). */
int glamr_opt_create(glamr_opt_t** out, const glamr_smpl_t* smpl, const glamr_problem_t* problem);
int glamr_opt_destroy(glamr_opt_t* st);
/* Re-read a modified problem description (new stage: weights, active mask, camera mode; same P, T, J, n_params).
 * reset_adam bit 0 zeroes the Adam moments and step count: the reference builds a fresh torch.optim.Adam per stage
 * (global_recon_model.py:548,:642); bit 1 also zeroes all scratch (handle re-used for a new sequence). */
int glamr_opt_set_problem(glamr_opt_t* st, const glamr_problem_t* problem, int reset_adam, void* stream);
/* length (floats) of the caller-owned reduce buffer: [grad (n_params) | un-normalised term sums (GLAMR_NUM_TERMS)] */
size_t glamr_opt_reduce_count(const glamr_opt_t* st);
/* kernels per optimiser iteration for the current problem (bench.py: gpu_launches), the same for a glamr_opt_iterate
 * loop and for a glamr_opt_backward + glamr_opt_apply pair */
int glamr_opt_launch_count(const glamr_opt_t* st);

/* forward (trajectory, camera, SMPL, projection) + residuals + analytic backward for the current theta, leaving
 * [grad | term sums] of THIS rank's share in reduce_buf.  With several GPUs the caller sums reduce_buf over ranks
 * (one NCCL allreduce) before glamr_opt_apply.  (closure of global_recon_model.py:551-557) */
int glamr_opt_backward(glamr_opt_t* st, const float* theta, float* reduce_buf, void* stream);
/* loss_terms [GLAMR_NUM_TERMS+1] (device): un-weighted term values (sum / normaliser) then the weighted total.
 * Then one torch.optim.Adam step (betas 0.9/0.999, eps 1e-8) on the active entries of theta; the step count and
 * bias corrections live on the device so the call sequence can be captured in a CUDA graph.  With
 * loss_hist_stride > 0 the terms of optimiser step k (0-based, counted on the device since the last reset) are
 * written at loss_terms + k * loss_hist_stride, so a replayed graph fills a per-iteration history. */
int glamr_opt_apply(glamr_opt_t* st, float* theta, const float* reduce_buf, double lr, float* loss_terms,
                    int loss_hist_stride, void* stream);
/* n_iters x (glamr_opt_backward + glamr_opt_apply) for a single-rank job (no reduction between the two).  With
 * use_graph != 0 the iteration is captured once into a CUDA graph owned by the handle (re-captured when the problem
 * or any argument changes) and replayed: the loop `for _ in range(opt_niters): optimizer.step(closure)` of
 * global_recon_model.py:558-569 becomes opt_niters graph launches with no host work in between. */
int glamr_opt_iterate(glamr_opt_t* st, float* theta, float* reduce_buf, double lr, float* loss_terms, int loss_hist_stride,
                      int n_iters, int use_graph, void* stream);
/* loss_terms only, no update (GlobalReconOptimizer.compute_loss, :533-545) */
int glamr_opt_losses(glamr_opt_t* st, const float* reduce_buf, float* loss_terms, void* stream);

/* Measurement hooks (bench.py roofline): when enabled, glamr_opt_backward brackets the LBS kernel with CUDA events on
 * the launching stream (do not enable while capturing a CUDA graph); glamr_opt_last_lbs_ms waits for the last pair
 * and returns its duration.  The only entry point that synchronises. */
/* glamr_opt_backward for a caller that runs glamr_opt_apply next on the same stream, with its exchange of reduce_buf in between (the
 * multi-GPU loop of global_recon_model.py:558-569): the pipelined side-stream work is joined by that apply call, not at the end of this one */
int glamr_opt_backward_for_apply(glamr_opt_t* st, const float* theta, float* reduce_buf, void* stream);
int glamr_opt_kernel_timing(glamr_opt_t* st, int enable);
/* the last timed evaluation split into the critical-path kernel (skinning; whole LBS kernel on the SIMT path) and the side-stream blend */
int glamr_opt_last_lbs_parts_ms(glamr_opt_t* st, float* critical_ms, float* blend_ms);
/* mean ms of the blend (feature kernel + tcgen05 GEMM) of this rank's frame-persons launched ALONE `reps` times (synchronises;
 * GLAMR_EUNSUPPORTED on the SIMT path or before the first evaluation) */
int glamr_opt_time_blend(glamr_opt_t* st, int reps, float* ms);
int glamr_opt_last_lbs_ms(glamr_opt_t* st, float* ms);
/* enable == 2: also record an event after every launch; durations (ms) between consecutive marks of the last
 * backward (+ apply) sequence: memset, traj_fwd, cam_fwd, pose_prep, lbs, joints, residuals, cam_bwd[, scatter], traj_bwd,
 * reduce[, losses, adam, advance] */
int glamr_opt_kernel_times(glamr_opt_t* st, float* ms, int* n);

enum glamr_read {
  GLAMR_R_ORIENT_WORLD = 0,    /* [P,T,3]   smpl_orient_world            */
  GLAMR_R_TRANS_WORLD = 1,     /* [P,T,3]   root_trans_world             */
  GLAMR_R_ORIENT_BASE = 2,     /* [P,T,3]   smpl_orient_world_base       */
  GLAMR_R_TRANS_BASE = 3,      /* [P,T,3]   root_trans_world_base        */
  GLAMR_R_KP_PRED = 4,         /* [P,T,J,2] kp_2d_pred                   */
  GLAMR_R_ORIENT_CAM_IN_WORLD = 5, /* [P,T,3]                            */
  GLAMR_R_TRANS_CAM_IN_WORLD = 6,  /* [P,T,3]                            */
  GLAMR_R_CAM_POSE = 7,        /* [T,12]    world->cam 3x4               */
  GLAMR_R_CAM_POSE_INV = 8,    /* [T,12]                                 */
  GLAMR_R_JOINTS_WORLD = 9,    /* [P,T,J,3]                              */
  GLAMR_R_TRAJ_LOCAL = 10      /* [P,T,11]  traj_local (rows of the exist range, others 0) */
};
/* ---- multi-GPU without a library collective: gradient reduction over NVLink peer memory --------------------------
 * One process per GPU.  Every rank allocates one buffer (glamr_peer_alloc; size glamr_opt_peer_bytes), ships its
 * 64-byte CUDA IPC handle to the other ranks (any host channel, e.g. torch.distributed.all_gather_object), opens theirs
 * (glamr_peer_open) and registers the table with glamr_opt_set_peers.  From then on, inside glamr_opt_iterate, the
 * backward pass pushes every element of [grad | term sums], tagged with the iteration number in the same 8-byte word,
 * into every rank's buffer, and the Adam kernel polls its own memory until the W tagged values of an element have
 * landed and sums them in rank order (identical bits on every rank): the all-reduce of global_recon's shared camera
 * gradient (SURVEY.md 8e) is fused into the Adam kernel -- no NCCL call, no fences, no host involvement, the whole
 * loop stays one replayed CUDA graph.  The stand-alone
 * glamr_opt_backward / glamr_opt_apply never touch peer memory (the caller reduces reduce_buf between them).
 * world <= 1 clears the table.  All ranks must call glamr_opt_iterate with the same iteration counts; a rank that
 * waits ~20 s for a peer traps (CUDA error) instead of hanging. */
#define GLAMR_MAX_PEERS 8
int glamr_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* ipc_handle_64_bytes);
int glamr_peer_open(const unsigned char* ipc_handle_64_bytes, void** dev_ptr);
int glamr_peer_close(void* dev_ptr);      /* a pointer from glamr_peer_open */
int glamr_peer_free(void* dev_ptr);       /* a pointer from glamr_peer_alloc */
size_t glamr_opt_peer_bytes(const glamr_opt_t* st);
int glamr_opt_set_peers(glamr_opt_t* st, int rank, int world, void* const* bufs /* [world], own buffer included */);
/* buf[0..count) <- element-wise sum over all ranks, in place, over the registered peer buffers (one kernel: every thread pushes
 * its elements to every rank, then polls its own buffer; count <= glamr_opt_reduce_count).  Collective: every rank calls it at the
 * same point of its stream order.  No-op for a single rank.  (SURVEY.md 8b `allreduce_inplace`; the per-iteration reduction of
 * glamr_opt_iterate is the same protocol fused into the Adam kernel.) */
int glamr_allreduce_inplace(glamr_opt_t* st, float* buf, size_t count, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Evaluation  --  stands behind global_recon/utils/evaluator.py:202-327 (Evaluator.prepare_seq).
 * glamr_sparse_regress: out[n,rows,3] = R @ vertices[n,V,3] for a regressor given in CSR form (row_ptr [rows+1], col_idx /
 *   weights [nnz], all DEVICE pointers) -- `torch.matmul(self.J_regressor, smpl_motion.vertices)` (:263,:306); the H36M
 *   regressor holds ~6 non-zeros per row.
 * glamr_procrustes_align: per frame, the similarity transform (scale, R, t) that maps S1 [n,J,3] closest to S2 [n,J,3],
 *   applied to S1 -> out [n,J,3]  (lib/utils/torch_transform.py:282-345 batch_compute_similarity_transform_torch; 3x3 SVD
 *   by one-sided Jacobi in fp64, reflection fixed through sign(det(U V^T))).
 * ---------------------------------------------------------------------------------------------------------- */
int glamr_sparse_regress(int n, int V, int rows, const int32_t* row_ptr, const int32_t* col_idx, const float* weights,
                         const float* vertices, float* out, void* stream);
int glamr_procrustes_align(int n, int J, const float* S1, const float* S2, float* out, void* stream);

/* device pointer + element count of an internal output buffer (valid until the handle is destroyed) */
int glamr_opt_read(glamr_opt_t* st, int what, const float** ptr, size_t* count);

#ifdef __cplusplus
}
#endif
#endif /* GLAMR_B200_H */
