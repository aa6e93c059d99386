"""Generate the golden fixtures under tests/golden/ by EXECUTING THE UNMODIFIED REFERENCE (/root/reference)
through the import shims of oracle/refshim (SURVEY.md Appendix C).  Run in the build container only:

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz and configs.json
    python tests/golden/make_golden.py configs    # only configs.json (the reference's shipped YAML configs)

The reference ships no tests and no golden vectors (SURVEY.md §4), so these outputs of the reference itself are
what pins the oracle (tests/test_oracle_vs_golden.py) and, through it, the CUDA path.  Inputs are regenerated
from seeds by glamr_b200.synthetic; only reference OUTPUTS (plus the learned-prior outputs that seed init_data)
are stored, so the fixtures stay small.
"""
import copy
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)

from oracle.refshim import ref_env  # noqa: E402

ref_env.activate(asset_seed=0)
import torch  # noqa: E402

from glamr_b200.synthetic import make_smpl_assets, make_in_dict  # noqa: E402

# (name, cfg, persons, frames, gaps, iterations per stage)
GLOBALOPT_CASES = [
    ('dynamic_p1_t40', 'glamr_dynamic', 1, 40, False, 6),
    ('static_p1_t24', 'glamr_static', 1, 24, False, 4),
    ('static_multi_p3_t30', 'glamr_static_multi', 3, 30, False, 5),
    ('dynamic_multi_p2_t32', 'glamr_dynamic_multi', 2, 32, False, 4),
    ('3dpw_p2_t80_gaps', 'glamr_3dpw', 2, 80, True, 4),
    ('h36m_p1_t48_gaps', 'glamr_h36m', 1, 48, True, 4),
    # the shapes bench.py measures (BASELINE.json configs[1], the north-star 4 x 300 video, T = 500 of configs[3]) and a
    # T > 512 track with gaps (more than one chunk of the CTA-wide prefix scans)
    ('dynamic_p1_t300', 'glamr_dynamic', 1, 300, False, 50),
    ('static_multi_p4_t300', 'glamr_static_multi', 4, 300, False, 10),
    ('static_multi_p2_t500', 'glamr_static_multi', 2, 500, False, 5),
    ('3dpw_p1_t600_gaps', 'glamr_3dpw', 1, 600, True, 4),
]
FINAL_KEYS = ['smpl_orient_world', 'root_trans_world', 'kp_2d_pred', 'traj_local_xy', 'traj_local_dxy', 'traj_local_heading',
              'traj_local_dheading', 'traj_local_z', 'traj_local_rot', 'world_dheading', 'smpl_orient_cam_in_world',
              'root_trans_cam_in_world', 'person_transform_world', 'traj_local']
FINAL_GLOBAL_KEYS = ['cam_pose', 'cam_pose_inv', 'cam_rot_6d', 'cam_trans', 'cam_rot_6d_fix', 'cam_trans_fix',
                     'cam_inv_rot_residual', 'cam_inv_trans_residual']


def float64_trajectory(assets, name, cfg_id, P, T, gaps, niters, rec):
    """Noise floor of the k-step comparison: the oracle restatement (pinned to the reference by
    tests/test_oracle_vs_golden.py) continues from the same float32 init state with every per-iteration formula in
    float64.  |final - final64| of the executed float32 reference is how far rounding noise alone moves the optimiser;
    the CUDA path is held to a small multiple of it (tests/test_gpu_parity.py)."""
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    from helpers import ReplayMT
    from glamr_b200.config import Config
    from oracle.global_opt import OracleGlobalRecon
    cfg = Config(cfg_id)
    for st in cfg.opt_stage_specs.values():
        st['opt_niters'] = niters
    in_dict = make_in_dict(assets, P, T, seed=0, gaps=gaps, seq_name=name)
    ora = OracleGlobalRecon(cfg, assets, mt_model=ReplayMT(rec))
    data = ora.to_float64(ora.init_data(in_dict))
    out = {}
    for stage, specs in cfg.opt_stage_specs.items():
        logs = []
        ora.optimize_main(data, specs['opt_variables'], specs['opt_lr'], specs['opt_niters'], specs['loss_cfg'], {'stage': stage},
                          on_iter=lambda it, last, dt: logs.append({k: float(v) for k, v in last['uw'].items()}))
        if specs.get('reinitialize_cam', False):
            from oracle import rotations as rt
            data['cam_pose'][:] = data['cam_pose'][[0]]
            data['cam_pose_inv'] = rt.inverse_transform(data['cam_pose'])
        for k in logs[0]:
            out[f'loss64/{stage}/{k}'] = np.asarray([l[k] for l in logs], np.float64)
    for k in FINAL_GLOBAL_KEYS:
        if k in data:
            out[f'final64/{k}'] = data[k].detach().numpy()
    for pid, pd in data['person_data'].items():
        for k in FINAL_KEYS:
            if k in pd and pd[k] is not None:
                out[f'final64/{pid}/{k}'] = pd[k].detach().numpy()
    out.update(perturbed_trajectory(assets, name, cfg_id, P, T, gaps, niters, rec))
    return out


def perturbed_trajectory(assets, name, cfg_id, P, T, gaps, niters, rec):
    """Second yardstick: the float32 oracle started from an init state whose float tensors are perturbed by ONE float32 rounding
    (x -> x (1 +- 2^-23), seeded signs).  Any re-implementation reaches the loop with such differences (sin/cos of another libm,
    another summation order); Adam's m / sqrt(v) turns a relative gradient change eps into parameter changes of ~ lr * k * eps.
    |final_pert - final| is that amplification measured on the reference's own arithmetic."""
    from helpers import ReplayMT
    from glamr_b200.config import Config
    from oracle.global_opt import OracleGlobalRecon
    cfg = Config(cfg_id)
    for st in cfg.opt_stage_specs.values():
        st['opt_niters'] = niters
    in_dict = make_in_dict(assets, P, T, seed=0, gaps=gaps, seq_name=name)
    ora = OracleGlobalRecon(cfg, assets, mt_model=ReplayMT(rec))
    data = ora.init_data(in_dict)
    g = torch.Generator().manual_seed(12345)

    def perturb(x):
        if isinstance(x, torch.Tensor) and x.dtype == torch.float32:
            sign = (torch.randint(0, 2, x.shape, generator=g).float() * 2 - 1)
            return x * (1 + sign * 2.0 ** -23)
        if isinstance(x, dict):
            return {k: perturb(v) for k, v in x.items()}
        return x
    data = perturb(data)
    out = {}
    for stage, specs in cfg.opt_stage_specs.items():
        logs = []
        ora.optimize_main(data, specs['opt_variables'], specs['opt_lr'], specs['opt_niters'], specs['loss_cfg'], {'stage': stage},
                          on_iter=lambda it, last, dt: logs.append({k: float(v) for k, v in last['uw'].items()}))
        if specs.get('reinitialize_cam', False):
            from oracle import rotations as rt
            data['cam_pose'][:] = data['cam_pose'][[0]]
            data['cam_pose_inv'] = rt.inverse_transform(data['cam_pose'])
        for k in logs[0]:
            out[f'loss_pert/{stage}/{k}'] = np.asarray([l[k] for l in logs], np.float64)
    for k in FINAL_GLOBAL_KEYS:
        if k in data:
            out[f'final_pert/{k}'] = data[k].detach().numpy()
    for pid, pd in data['person_data'].items():
        for k in FINAL_KEYS:
            if k in pd and pd[k] is not None:
                out[f'final_pert/{pid}/{k}'] = pd[k].detach().numpy()
    return out



def rotation_vectors():
    """Function-level known answers for the rotation algebra, including the branch points (zero angle, theta^2
    below 1e-6, trace<=0 quaternion branches, w<0) -- SURVEY.md §7 'hard parts'."""
    from lib.utils import konia_transform as K
    from lib.utils import torch_transform as TT
    g = torch.Generator().manual_seed(7)
    aa = torch.randn(48, 3, generator=g)
    aa[:4] = 0.0
    aa[4:8] *= 1e-4                                   # theta^2 < 1e-6 -> taylor / clamp branches
    aa[8:12] *= 3e-3
    aa[12:16] = torch.nn.functional.normalize(aa[12:16], dim=-1) * 3.1
    aa[16] = torch.tensor([0.0, 0.0, 0.3])
    d6 = torch.randn(48, 6, generator=g)
    R = K.angle_axis_to_rotation_matrix(aa)
    big = torch.nn.functional.normalize(torch.randn(24, 3, generator=g), dim=-1) * torch.linspace(2.4, 3.14, 24)[:, None]
    Rbig = K.angle_axis_to_rotation_matrix(big)       # trace <= 0 -> the three non-trace quaternion branches
    Rall = torch.cat([R, Rbig])
    q = torch.randn(48, 4, generator=g)
    q[:8] = torch.nn.functional.normalize(q[:8], dim=-1)
    q[8] = torch.tensor([1.0, 0.0, 0.0, 0.0])
    q[9] = torch.tensor([-1.0, 0.0, 0.0, 0.0])
    q[10] = torch.tensor([0.0, 0.0, 0.0, 1.0])
    q[11] = torch.tensor([0.9999999, 1e-4, 0.0, 0.0])
    qn = torch.nn.functional.normalize(q, dim=-1)
    q2 = torch.nn.functional.normalize(torch.randn(48, 4, generator=g), dim=-1)
    y = torch.randn(48, generator=g)
    x = torch.randn(48, generator=g)
    y[:4], x[:4] = 0.0, 0.0
    y[4:8], x[4:8] = 1e-7, -1e-7
    out = {
        'in_aa': aa, 'in_d6': d6, 'in_R': Rall, 'in_q': q, 'in_qn': qn, 'in_q2': q2, 'in_y': y, 'in_x': x,
        'aa_to_rotmat': K.angle_axis_to_rotation_matrix(aa),
        'rotmat_to_quat': K.rotation_matrix_to_quaternion(Rall.contiguous()),
        'quat_to_aa': K.quaternion_to_angle_axis(qn),
        'quat_to_aa_raw': K.quaternion_to_angle_axis(q),
        'aa_to_quat': K.angle_axis_to_quaternion(aa),
        'quat_to_rotmat': K.quaternion_to_rotation_matrix(q),
        'rotmat_to_aa': K.rotation_matrix_to_angle_axis(Rall.contiguous()),
        'quat_mul': TT.quat_mul(qn, q2),
        'quat_angle_diff': TT.quat_angle_diff(qn, q2),
        'safe_atan2': TT.torch_safe_atan2(y, x),
        'rot6d_to_rotmat': TT.rot6d_to_rotmat(d6),
        'aa_to_rot6d': TT.angle_axis_to_rot6d(aa),
        'rot6d_to_quat': TT.rot6d_to_quat(d6),
        'get_heading': TT.get_heading(qn),
        'get_heading_q': TT.get_heading_q(qn),
        'heading_to_quat': TT.heading_to_quat(y),
        'deheading_quat': TT.deheading_quat(qn),
    }
    M = TT.make_transform(aa, d6[:, :3], rot_type='axis_angle')
    out['make_transform_aa'] = M
    out['inverse_transform'] = TT.inverse_transform(M)
    out['transform_rot'] = TT.transform_rot(M, aa.flip(0))
    out['transform_trans'] = TT.transform_trans(M, d6[:, 3:])
    # docstring known answer of the reference (konia_transform.py:492-497)
    out['doc_quat_to_rotmat'] = K.quaternion_to_rotation_matrix(torch.tensor((0., 0., 0., 1.)))
    return {k: v.numpy() for k, v in out.items()}


def traj_vectors():
    from traj_pred.utils import traj_utils as TU
    from lib.utils import torch_transform as TT
    g = torch.Generator().manual_seed(11)
    T = 37
    local = torch.randn(T, 11, generator=g) * 0.3
    local[:, 3:9] += torch.tensor([1.0, 0, 0, 0, 1.0, 0])
    local[:, -2:] = torch.nn.functional.normalize(torch.randn(T, 2, generator=g), dim=-1)
    trans, q = TU.traj_local2global_heading(local)
    back = TU.traj_global2local_heading(trans, q)
    vis = torch.ones(T, dtype=torch.bool)
    vis[5:11] = False
    vis[20:23] = False
    qi = TU.interp_orient_q_sep_heading(q[vis], vis)
    return {'in_local': local.numpy(), 'trans': trans.numpy(), 'orient_q': q.numpy(), 'orient_aa': TT.quaternion_to_angle_axis(q).numpy(),
            'global_to_local': back.numpy(), 'in_vis': vis.numpy(), 'interp_q': qi.numpy()}


def smpl_vectors(assets):
    from lib.models.smpl import SMPL, SMPL_MODEL_DIR
    smpl = SMPL(SMPL_MODEL_DIR, pose_type='body26fk', create_transl=False)
    g = torch.Generator().manual_seed(3)
    B = 9
    orient = torch.randn(B, 3, generator=g)
    pose = torch.randn(B, 69, generator=g) * 0.3
    pose[0] = 0.0
    orient[0] = 0.0
    betas = torch.randn(B, 10, generator=g)
    trans = torch.randn(B, 3, generator=g)
    scale = torch.rand(B, generator=g) + 0.5
    o = smpl(global_orient=orient, body_pose=pose, betas=betas, root_trans=trans, root_scale=None, return_full_pose=True)
    o_s = smpl(global_orient=orient, body_pose=pose, betas=betas, root_trans=trans, root_scale=scale, return_full_pose=True)
    o_raw = smpl(global_orient=orient, body_pose=pose, betas=betas, return_full_pose=True)
    o_24 = smpl(global_orient=orient, body_pose=pose, betas=betas, root_trans=trans, orig_joints=True)
    fk = smpl.get_joints(body_pose=pose, global_orient=orient, root_trans=trans)
    vsel = np.arange(0, 6890, 53)
    return {
        'in_orient': orient.numpy(), 'in_pose': pose.numpy(), 'in_betas': betas.numpy(), 'in_trans': trans.numpy(),
        'in_scale': scale.numpy(), 'vsel': vsel,
        'joints': o.joints.numpy(), 'verts_sel': o.vertices[:, vsel].numpy(), 'verts_sum': o.vertices.double().sum(1).numpy(),
        'verts_abs_sum': o.vertices.double().abs().sum(1).numpy(),
        'joints_scaled': o_s.joints.numpy(), 'verts_scaled_sel': o_s.vertices[:, vsel].numpy(),
        'joints_raw': o_raw.joints.numpy(), 'verts_raw_sel': o_raw.vertices[:, vsel].numpy(),
        'joints24': o_24.joints.numpy(), 'verts24_sel': o_24.vertices[:, vsel].numpy(),
        'fk_joints': fk.numpy(),
    }


def nets_vectors():
    """MotionTrajJointModel.inference of the reference with the seeded stand-in weights of
    glamr_b200.synthetic_nets loaded into its modules, latents injected (CPU and CUDA generators differ)."""
    from motion_infiller.models.motion_traj_joint_model import MotionTrajJointModel
    from motion_infiller.utils.config_motion_traj import Config as MTConfig
    from glamr_b200.synthetic_nets import make_prior_states
    mt = MotionTrajJointModel(MTConfig('joint_motion_traj_demo'), torch.device('cpu'), None)
    st_m, st_t = make_prior_states(1234)
    for mod, st in [(mt.mfiller, st_m), (mt.traj_predictor, st_t)]:
        own = mod.state_dict()
        assert all(k in own and tuple(own[k].shape) == v.shape for k, v in st.items()), 'state-dict names/shapes differ from the reference'
        res = mod.load_state_dict({k: torch.tensor(v) for k, v in st.items()}, strict=False)
        assert not res.unexpected_keys
    out = {}
    g = torch.Generator().manual_seed(21)
    for tag, B, T in [('b3_t75', 3, 75), ('b1_t300', 1, 300), ('b2_t40', 2, 40)]:
        pose = torch.randn(B, T, 69, generator=g) * 0.3
        mask = torch.ones(B, T)
        mask[0, 20:45] = 0
        if B > 1:
            mask[1, T - 12:T - 2] = 0
        nwin = int(np.ceil((T - 10) / 30))
        batch = {'in_body_pose': pose * mask[..., None], 'frame_mask': mask, 'in_motion_latent': torch.randn(nwin, 128, generator=g),
                 'in_traj_latent': torch.randn(1, 128, generator=g)}
        res = mt.inference({k: v.clone() for k, v in batch.items()}, sample_num=1)
        for k, v in batch.items():
            out[f'{tag}/in/{k}'] = v.numpy()
        for k in ['infer_out_body_pose', 'infer_out_local_traj_tp', 'infer_out_orient', 'infer_out_trans', 'infer_out_pose']:
            out[f'{tag}/{k}'] = res[k].detach().numpy()
    # BASELINE.json configs[2]: batch 64 x 120 frames, frames 40-69 masked.  Inputs are regenerated from the seed by
    # c3_prior_inputs() (shared with the GPU test); stored: four whole sequences and per-sequence sums of all 64.
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    from helpers import C3_ROWS, c3_prior_inputs
    batch = c3_prior_inputs()
    res = mt.inference({k: v.clone() for k, v in batch.items()}, sample_num=1)
    sel = C3_ROWS
    for k, bdim in [('infer_out_body_pose', 0), ('infer_out_local_traj_tp', 1), ('infer_out_orient', 0), ('infer_out_trans', 0)]:
        v = res[k].detach()
        out[f'c3_b64_t120/{k}'] = v.index_select(bdim, torch.tensor(sel)).numpy()
        red = [d for d in range(v.dim()) if d != bdim]
        out[f'c3_b64_t120/{k}/sum'] = v.double().sum(dim=red).numpy()
        out[f'c3_b64_t120/{k}/abs_sum'] = v.double().abs().sum(dim=red).numpy()
    return out


def nets_c3_float64_vectors():
    """The C3-shape run of nets_vectors with the reference networks, its SMPL and the inputs in float64 (default dtype float64
    while the reference builds and runs, so that the state its modules create is float64 too): per-sequence sums of all 64
    sequences.  The trajectory is integrated over 120 frames; with the seeded stand-in weights the heading reaches a few
    hundred radians, where one float32 ulp is 3e-5 rad, so float32 sums differ from host to host (thread count, SIMD width)
    by more than the 1e-5 the oracle is held to.  In float64 they do not."""
    from motion_infiller.models.motion_traj_joint_model import MotionTrajJointModel
    from motion_infiller.utils.config_motion_traj import Config as MTConfig
    from glamr_b200.synthetic_nets import make_prior_states
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    from helpers import c3_prior_inputs
    batch = {k: v.double() if v.is_floating_point() else v for k, v in c3_prior_inputs().items()}   # drawn in float32, as the tests draw them
    torch.set_default_dtype(torch.float64)
    try:
        mt = MotionTrajJointModel(MTConfig('joint_motion_traj_demo'), torch.device('cpu'), None)
        st_m, st_t = make_prior_states(1234)
        for mod, st in [(mt.mfiller, st_m), (mt.traj_predictor, st_t)]:
            res = mod.load_state_dict({k: torch.tensor(v) for k, v in st.items()}, strict=False)
            assert not res.unexpected_keys
        for mod in (mt.mfiller, mt.traj_predictor, mt.smpl):          # buffers loaded from float32 files (the SMPL models)
            mod.double()
        res = mt.inference(batch, sample_num=1)
    finally:
        torch.set_default_dtype(torch.float32)
    out = {}
    for k, bdim in [('infer_out_body_pose', 0), ('infer_out_local_traj_tp', 1), ('infer_out_orient', 0), ('infer_out_trans', 0)]:
        v = res[k].detach()
        assert v.dtype == torch.float64, k
        red = [d for d in range(v.dim()) if d != bdim]
        out[f'c3_b64_t120/{k}/sum'] = v.sum(dim=red).numpy()
        out[f'c3_b64_t120/{k}/abs_sum'] = v.abs().sum(dim=red).numpy()
    return out


def globalopt_case(assets, name, cfg_id, P, T, gaps, niters):
    in_dict = make_in_dict(assets, P, T, seed=0, gaps=gaps, seq_name=name)
    model, cfg = ref_env.make_reference_optimizer(cfg_id, niters=niters)
    rec = {}
    # 1) learned-prior outputs per person (the nets here are seeded random-init; the fixtures replay them)
    mt_calls = []
    orig_inf = model.mt_model.inference

    def rec_inference(batch, sample_num=1):
        out = orig_inf(batch, sample_num=sample_num)
        mt_calls.append({k: out[k].detach().clone() for k in
                         ['infer_out_body_pose', 'infer_out_local_traj_tp', 'infer_out_orient', 'infer_out_trans']})
        return out
    model.mt_model.inference = rec_inference
    # 2) per-iteration unweighted residuals + iteration-0 gradients of every stage
    state = {'params': None}
    orig_init_opt = model.init_opt

    def rec_init_opt(data, opt_variables, opt_lr):
        opt, params = orig_init_opt(data, opt_variables, opt_lr)
        state['params'] = params
        return opt, params
    model.init_opt = rec_init_opt
    losses = {}

    def rec_logs(loss_dict, meta):
        st, it = meta['stage'], meta['cur_iter']
        for k, v in loss_dict.items():
            losses.setdefault(f'{st}/{k}', []).append(float(v))
        if it == 0:
            for i, p in enumerate(state['params']):
                # a parameter autograd never reached has grad None (Adam skips it): stored as an empty array
                rec[f'grad0/{st}/{i}'] = (p.grad.detach().clone().numpy() if p.grad is not None else np.zeros((0,), np.float32))
                rec[f'param_shape/{st}/{i}'] = np.asarray(p.shape)
    model.write_logs = rec_logs
    # 3) state right after init_data
    orig_init = model.init_data

    def rec_init(d):
        data = orig_init(d)
        for pid, pd in data['person_data'].items():
            for k in ['kp_2d_pred', 'smpl_orient_world', 'root_trans_world', 'traj_local_pred', 'smpl_pose', 'vis_frames',
                      'smpl_orient_cam', 'root_trans_cam', 'person2cam']:
                rec[f'init/{pid}/{k}'] = pd[k].detach().clone().numpy()
        rec['init/cam_pose'] = data['cam_pose'].detach().clone().numpy()
        return data
    model.init_data = rec_init
    torch.manual_seed(0)
    out = model.optimize(copy.deepcopy(in_dict))
    for i, c in enumerate(mt_calls):
        for k, v in c.items():
            rec[f'mt/{i}/{k}'] = v.numpy()
    for k, v in losses.items():
        rec[f'loss/{k}'] = np.asarray(v, np.float64)
    for k in FINAL_GLOBAL_KEYS:
        if k in out:
            rec[f'final/{k}'] = out[k]
    for pid, pd in out['person_data'].items():
        for k in FINAL_KEYS:
            if k in pd and pd[k] is not None:
                rec[f'final/{pid}/{k}'] = pd[k]
    rec['meta'] = np.array([P, T, int(gaps), niters])
    rec['cfg_id'] = np.array(cfg_id)
    rec.update(float64_trajectory(assets, name, cfg_id, P, T, gaps, niters, rec))
    return rec


def camera_term_vectors():
    """camera-only residuals that no shipped config enables (so the global-opt fixtures never exercise them), evaluated
    by the reference's own functions on a seeded camera track"""
    from global_recon.models import loss_func as ref_loss
    from lib.utils.torch_transform import make_transform
    g = torch.Generator().manual_seed(5)
    T = 37
    rot6d = torch.tensor([1., 0., 0., 0., 1., 0.]) + 0.2 * torch.randn(T, 6, generator=g)
    trans = torch.cumsum(0.05 * torch.randn(T, 3, generator=g), dim=0)
    inv = make_transform(rot6d, trans, rot_type='6d')
    data = {'cam_pose_inv': inv}
    rec = {'cam_rot6d': rot6d.numpy(), 'cam_trans': trans.numpy(), 'cam_pose_inv': inv.numpy()}
    for name in ['cam_depth_smoothness', 'cam_origin_smoothness', 'cam_inv_rot_smoothness']:
        rec[name] = np.asarray(float(ref_loss.loss_func_dict[name](data, {})))
    return rec


def evaluator_vectors():
    """Evaluator.compute_sequence_metrics of the reference (global_recon/utils/evaluator.py) on seeded (estimate, ground truth)
    pairs.  The reference imports `lib.utils.logging`, a module its tree does not contain (the file is lib/utils/log_utils.py):
    aliased in sys.modules, like the other import shims; its code is untouched."""
    import lib.utils.log_utils as LU
    sys.modules['lib.utils.logging'] = LU
    from glamr_b200.synthetic import make_eval_case, make_h36m_regressor
    np.save(os.path.join(ref_env.WORK, 'data', 'J_regressor_h36m.npy'), make_h36m_regressor(0))
    from global_recon.utils.evaluator import Evaluator
    out = {}
    for tag, dataset, P, T, freq in [('p2_t60', '3DPW', 2, 60, 250), ('p1_t300_h36m', 'h36m', 1, 300, 250), ('p1_t90_realign', '3DPW', 1, 90, 40)]:
        ev = Evaluator('glamr', dataset, device=torch.device('cpu'), log_file='nofile', align_freq=freq, compute_sample=True)
        data = make_eval_case(P, T, seed=len(out))
        out[f'{tag}/seed'] = np.array(len(out))
        md = ev.compute_sequence_metrics(copy.deepcopy(data), 'case', accumulate=False)
        for k, v in md['metrics'].items():
            if isinstance(v.avg, np.ndarray):
                out[f'{tag}/metric/{k}'] = v.avg
            else:
                out[f'{tag}/metric/{k}'] = np.array([v.avg, v.count], np.float64)
    return out


def config_vectors():
    """the six shipped configs of the reference (global_recon/cfg/<id>.yml) as parsed by yaml.safe_load: the stage / weight
    tables that glamr_b200.config.builtin_config_dict rebuilds"""
    import yaml
    from glamr_b200.config import BUILTIN_IDS
    out = {}
    for cfg_id in BUILTIN_IDS:
        with open(os.path.join(ref_env.REF_ROOT, 'global_recon', 'cfg', cfg_id + '.yml')) as f:
            d = yaml.safe_load(f)
        out[cfg_id] = {k: d[k] for k in ['grecon_model_name', 'dataset', 'grecon_model_specs', 'opt_stage_specs']}
    return out


def write_configs():
    with open(os.path.join(HERE, 'configs.json'), 'w') as f:
        json.dump(config_vectors(), f, indent=1, sort_keys=True)


def main(only=None):
    if only == 'configs':
        write_configs()
        return
    if only == 'evaluator':
        np.savez_compressed(os.path.join(HERE, 'evaluator.npz'), **evaluator_vectors())
        return
    if only == 'camera_terms':
        np.savez_compressed(os.path.join(HERE, 'camera_terms.npz'), **camera_term_vectors())
        return
    if only == 'nets':
        np.savez_compressed(os.path.join(HERE, 'nets.npz'), **nets_vectors())
        np.savez_compressed(os.path.join(HERE, 'nets_c3_f64.npz'), **nets_c3_float64_vectors())
        return
    if only == 'nets_c3_f64':
        np.savez_compressed(os.path.join(HERE, 'nets_c3_f64.npz'), **nets_c3_float64_vectors())
        return
    assets = make_smpl_assets(0)
    if only is not None:                       # one global-opt case by name (adding a fixture without touching the others)
        case = [c for c in GLOBALOPT_CASES if c[0] == only][0]
        np.savez_compressed(os.path.join(HERE, f'globalopt_{case[0]}.npz'), **globalopt_case(assets, *case))
        print('wrote', case[0])
        return
    write_configs()
    np.savez_compressed(os.path.join(HERE, 'rotations.npz'), **rotation_vectors())
    np.savez_compressed(os.path.join(HERE, 'traj_codec.npz'), **traj_vectors())
    np.savez_compressed(os.path.join(HERE, 'smpl.npz'), **smpl_vectors(assets))
    np.savez_compressed(os.path.join(HERE, 'nets.npz'), **nets_vectors())
    np.savez_compressed(os.path.join(HERE, 'nets_c3_f64.npz'), **nets_c3_float64_vectors())
    for case in GLOBALOPT_CASES:
        rec = globalopt_case(assets, *case)
        np.savez_compressed(os.path.join(HERE, f'globalopt_{case[0]}.npz'), **rec)
        print('wrote', case[0], len(rec), 'arrays')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else None)
