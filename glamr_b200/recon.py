"""``GlobalReconOptimizer`` -- drop-in for the reference class of the same name
(global_recon/models/global_recon_model.py:23-659) with the optimisation loop running in the CUDA library.

Same constructor, ``optimize(in_dict, continue_opt=False) -> dict`` (numpy), ``init_data``, ``forward``,
``compute_loss``, ``optimize_main``; same YAML stage specs; same output keys / shapes / dtypes (SURVEY.md Appendix B).
Host Python does what the reference does on the host (dict bookkeeping, SciPy rotation-vector conversion and linear
gap interpolation, log lines); every formula of the per-iteration path -- trajectory codec, camera, SMPL, projection,
residuals, analytic backward, Adam -- is a kernel of glamr_b200/csrc.  No autograd, no CPU fallback.
"""
import ctypes
import time

import numpy as np
import torch
from scipy.interpolate import interp1d

from . import geometry as G
from . import lib as L
from . import problem as PB
from .smpl import SMPL, SMPL_MODEL_DIR
from .synthetic import SMPL_TO_BODY26FK

NUM_TERMS = L.NUM_TERMS
_TERM_NAMES = {v: k for k, v in L.TERM_INDEX.items()}


def tensor_to(x, device):
    """lib/utils/torch_utils.py:101 -- numpy / nested containers -> tensors on `device` (dtype preserved)"""
    if isinstance(x, np.ndarray):
        return torch.tensor(x, device=device)
    if isinstance(x, torch.Tensor):
        return x.to(device)
    if isinstance(x, dict):
        return {k: tensor_to(v, device) for k, v in x.items()}
    return x


_GROUP_CPU_TENSORS = False      # tests flip this to run the grouped-copy path on CPU tensors


def tensor_to_numpy(x):
    """lib/utils/torch_utils.py:118 -- nested containers of tensors -> numpy.  The output dict of `optimize` holds several
    hundred small tensors per person; instead of one synchronous device->host copy each, the tensors of one dtype are
    concatenated on the device, copied once and split into views on the host (same values, shapes and dtypes)."""
    leaves = []

    def walk(v):
        if isinstance(v, torch.Tensor):
            leaves.append(v.detach())
            return ('leaf', len(leaves) - 1)
        if isinstance(v, dict):
            return ('dict', {k: walk(u) for k, u in v.items()})
        if isinstance(v, (list, tuple)):
            return (type(v), [walk(u) for u in v])
        return ('raw', v)
    tree = walk(x)
    arrays = [None] * len(leaves)
    groups = {}
    for i, t in enumerate(leaves):
        groups.setdefault((t.dtype, t.device), []).append(i)
    for (dtype, device), idx in groups.items():
        if len(idx) == 1 or (device.type == 'cpu' and not _GROUP_CPU_TENSORS):
            for i in idx:
                arrays[i] = leaves[i].cpu().numpy()
            continue
        flat = torch.cat([leaves[i].reshape(-1) for i in idx]).cpu().numpy()
        off = 0
        for i in idx:
            n = leaves[i].numel()
            arrays[i] = flat[off:off + n].reshape(tuple(leaves[i].shape))
            off += n

    def build(node):
        kind, v = node
        if kind == 'leaf':
            return arrays[v]
        if kind == 'dict':
            return {k: build(u) for k, u in v.items()}
        if kind == 'raw':
            return v
        return kind(build(u) for u in v)
    return build(tree)


def rotmats_to_rotvec(mats):
    """``Rotation.from_matrix(mats).as_rotvec()`` (global_recon_model.py:106-107) as vectorised numpy, float64.

    SciPy projects every float32-accurate input onto SO(3) with one SVD per matrix (12 ms for a 300-frame track); the
    same polar factor U V^T is reached here by two Newton steps R <- (R + R^-T) / 2 written with cross products, then
    the usual largest-diagonal quaternion branch and the rotation-vector scaling (series below 1e-3 rad).  The nine
    entries are kept as nine contiguous arrays (structure of arrays): every step is a handful of long vector operations."""
    R0 = np.asarray(mats, dtype=np.float64).reshape(-1, 3, 3)
    n = R0.shape[0]
    r = np.ascontiguousarray(R0.reshape(n, 9).T)                      # r[3 i + j] = R[:, i, j], contiguous
    det = None
    for _ in range(2):
        a0, a1, a2, b0, b1, b2, c0, c1, c2 = r
        cof = np.empty_like(r)                                       # cofactor rows = cross products of the other two rows
        cof[0] = b1 * c2 - b2 * c1
        cof[1] = b2 * c0 - b0 * c2
        cof[2] = b0 * c1 - b1 * c0
        cof[3] = c1 * a2 - c2 * a1
        cof[4] = c2 * a0 - c0 * a2
        cof[5] = c0 * a1 - c1 * a0
        cof[6] = a1 * b2 - a2 * b1
        cof[7] = a2 * b0 - a0 * b2
        cof[8] = a0 * b1 - a1 * b0
        det = a0 * cof[0] + a1 * cof[1] + a2 * cof[2]
        with np.errstate(divide='ignore', invalid='ignore'):
            r = 0.5 * (r + cof / det)
    # two Newton steps reach the polar factor only from a near-orthogonal start (HybrIK's float32 matrices).  Rows that are
    # not there yet (or improper / singular inputs) go through SciPy's SVD projection like the reference (which also raises
    # on non-finite input).
    a0, a1, a2, b0, b1, b2, c0, c1, c2 = r
    resid = np.maximum.reduce([np.abs(a0 * a0 + a1 * a1 + a2 * a2 - 1), np.abs(b0 * b0 + b1 * b1 + b2 * b2 - 1), np.abs(c0 * c0 + c1 * c1 + c2 * c2 - 1),
                               np.abs(a0 * b0 + a1 * b1 + a2 * b2), np.abs(a0 * c0 + a1 * c1 + a2 * c2), np.abs(b0 * c0 + b1 * c1 + b2 * c2)])
    bad = ~(det > 0) | ~(resid < 1e-9)
    if bad.any():
        from scipy.spatial.transform import Rotation
        r = r.copy()
        r[:, bad] = Rotation.from_matrix(R0[bad]).as_matrix().reshape(-1, 9).T
        a0, a1, a2, b0, b1, b2, c0, c1, c2 = r
    tr = a0 + b1 + c2
    d = np.stack([a0, b1, c2, tr])
    choice = d.argmax(axis=0)
    q = np.empty((4, n))
    R = r.reshape(3, 3, n)
    for i in range(3):
        sel = np.where(choice == i)[0]
        if sel.size == 0:
            continue
        j, k = (i + 1) % 3, (i + 2) % 3
        q[i, sel] = 1 - tr[sel] + 2 * R[i, i, sel]
        q[j, sel] = R[j, i, sel] + R[i, j, sel]
        q[k, sel] = R[k, i, sel] + R[i, k, sel]
        q[3, sel] = R[k, j, sel] - R[j, k, sel]
    sel = np.where(choice == 3)[0]
    q[0, sel] = R[2, 1, sel] - R[1, 2, sel]
    q[1, sel] = R[0, 2, sel] - R[2, 0, sel]
    q[2, sel] = R[1, 0, sel] - R[0, 1, sel]
    q[3, sel] = 1 + tr[sel]
    q /= np.sqrt((q * q).sum(axis=0))
    q[:, q[3] < 0] *= -1
    angle = 2 * np.arctan2(np.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2]), q[3])
    small = angle <= 1e-3
    a2_ = angle * angle
    with np.errstate(divide='ignore', invalid='ignore'):
        scale = np.where(small, 2 + a2_ / 12 + 7 * a2_ * a2_ / 2880, angle / np.sin(angle / 2))
    return np.ascontiguousarray((scale * q[:3]).T)


def _sec_to_time(secs):
    secs = int(secs)
    return f'{secs // 3600}:{(secs % 3600) // 60:02d}:{secs % 60:02d}'


class GlobalReconOptimizer:

    def __init__(self, cfg, device=torch.device('cuda'), log=None, smpl=None, mt_model=None, dist=None):
        """cfg/device/log as in the reference (:25).  Extra, optional:
        smpl      a glamr_b200.smpl.SMPL (or an assets dict); default loads SMPL_MODEL_DIR like the reference
        mt_model  object with .inference(batch, sample_num) (the learned prior); default: the CUDA MotionTrajJointModel
        dist      (rank, world_size) for person sharding across GPUs (torch.distributed must be initialised)"""
        self.cfg = cfg
        self.specs = specs = cfg.grecon_model_specs
        self.device = L.require_cuda(device)
        self.log = log
        self.cur_iter = 0
        if isinstance(smpl, SMPL):
            self.smpl = smpl
        else:
            self.smpl = SMPL(smpl if smpl is not None else SMPL_MODEL_DIR, pose_type='body26fk', device=self.device)
        g = specs.get
        self.use_gt = g('use_gt', False)
        self.est_type = g('est_type', 'hybrik')
        self.flag_infer_motion_traj = g('flag_infer_motion_traj', False)
        self.flag_infill_motion = g('flag_infill_motion', True)
        self.flag_pred_traj = g('flag_pred_traj', True)
        self.flag_opt_traj = g('flag_opt_traj', True)
        self.flag_opt_cam = g('flag_opt_cam', True)
        self.flag_fixed_cam = g('flag_fixed_cam', False)
        self.flag_opt_vis_local_rot = g('flag_opt_vis_local_rot', False)
        self.flag_opt_person2cam_rot = g('flag_opt_person2cam_rot', False)
        self.flag_opt_person2cam_trans = g('flag_opt_person2cam_trans', False)
        self.flag_cam_inv_trans_res_all = g('flag_cam_inv_trans_res_all', True)
        self.flag_filter_pose = g('flag_filter_pose', True)
        self.flag_make_invis_with_keypoint = g('flag_make_invis_with_keypoint', False)
        self.make_invis_keypoint_min_score = g('make_invis_keypoint_min_score', 0.6)
        self.make_invis_keypoint_min_num = g('make_invis_keypoint_min_num', 15)
        self.flag_opt_cam_from_person_pose = g('flag_opt_cam_from_person_pose', False)
        self.flag_init_cam_all_frames = g('flag_init_cam_all_frames', False)
        self.cam_fix_frames = g('cam_fix_frames', [[0, None]])
        self.opt_stage_specs = self.cfg.opt_stage_specs
        for flag in ['flag_opt_motion_latent', 'flag_opt_traj_latent', 'flag_use_pen_loss', 'flag_traj_from_cam', 'absolute_heading']:
            if g(flag, False):
                raise NotImplementedError(f'{flag} is not implemented in the CUDA path (SURVEY.md §8(f)-4); no CPU fallback')
        if g('heading_type', 'scalar') != 'scalar':
            raise NotImplementedError("heading_type 'vec' is not implemented in the CUDA path")
        if not self.flag_opt_traj:
            raise NotImplementedError('flag_opt_traj=false is not implemented in the CUDA path')
        self.rank, self.world = dist if dist is not None else (0, 1)
        self.log_interval = g('log_interval', 1)
        self.use_cuda_graph = g('use_cuda_graph', True)
        self.mt_cfg = None
        self.mt_model = mt_model
        if mt_model is None and 'motion_traj_cfg' in specs and self.flag_infer_motion_traj:
            self.load_model()
        self._lib = L.load()
        self._opt = None
        self.iter_ms = []              # (stage, niters, ms per iteration) of every optimize_main call

    def load_model(self):
        from .motion_traj import MotionTrajJointModel
        self.mt_model = MotionTrajJointModel(self.specs['motion_traj_cfg'], self.device, self.log, smpl=self.smpl)
        self.mt_cfg = getattr(self.mt_model, 'cfg', None)

    @property
    def _flags(self):
        return {k: getattr(self, k) for k in ['flag_fixed_cam', 'flag_opt_cam', 'flag_opt_cam_from_person_pose',
                                              'flag_cam_inv_trans_res_all', 'flag_opt_vis_local_rot', 'cam_fix_frames',
                                              'flag_opt_person2cam_rot', 'flag_opt_person2cam_trans']}

    # ------------------------------------------------------------------------------------------------ init_data
    def _person_from_estimate(self, est, gt_entry):
        """global_recon_model.py:88-137 (host side, numpy/SciPy exactly as the reference)"""
        d = {}
        visible = est['bboxes_dict']['exist'].copy()
        d['visible'] = visible
        d['visible_orig'] = visible.copy()
        where = np.where(visible)[0]
        start, end = where[0], where[-1] + 1
        d['fr_start'], d['fr_end'] = start, end
        exist = visible == 1
        exist[start:end] = True
        d['exist_frames'] = exist
        d['exist_len'] = end - start
        d['max_len'] = n = visible.shape[0]
        d['frames'] = np.arange(n)
        d['vis_frames'] = vis = visible == 1
        d['invis_frames'] = visible == 0
        d['frame2ind'] = {f: i for i, f in enumerate(d['frames'])}
        d['scale'] = None
        rotmats = est['smpl_pose_quat_wroot']
        nv = rotmats.shape[0]
        aa = rotmats_to_rotvec(rotmats).reshape(nv, -1, 3).astype(np.float32)
        d['smpl_pose'] = aa[:, 1:].reshape(-1, 69)
        if gt_entry is not None:
            d['smpl_pose_gt'] = gt_entry['pose'][:, 3:]
        d['smpl_beta'] = est['smpl_beta']
        d['smpl_orient_cam'] = aa[:, 0]
        d['root_trans_cam'] = est['root_trans']
        j2d = est['kp_2d'][:, :24]
        j2d = np.concatenate([j2d, np.ones_like(j2d[:, :, :1])], axis=-1)
        kp = np.zeros((int(vis.sum()), 26, 3))
        kp[:, SMPL_TO_BODY26FK[:, 0]] = j2d[:, SMPL_TO_BODY26FK[:, 1]]
        d['kp_2d'], d['kp_2d_score'] = kp[:, :, :2], kp[:, :, 2]
        d['kp_2d_aligned'] = d['kp_2d'].copy()
        d['cam_K'] = est['cam_K'].astype(np.float32)
        if not np.all(visible):
            for key in ['kp_2d', 'kp_2d_score', 'kp_2d_aligned', 'cam_K']:
                full = np.zeros((n,) + d[key].shape[1:], dtype=d[key].dtype)
                full[vis] = d[key]
                d[key] = full
            vis_ind = np.where(visible)[0].astype(np.float32)
            for key in ['smpl_pose', 'smpl_beta', 'root_trans_cam', 'smpl_orient_cam']:
                f = interp1d(vis_ind, d[key], axis=0, assume_sorted=True, fill_value='extrapolate')
                d[key] = f(np.arange(n, dtype=np.float32))
        return tensor_to(d, self.device)

    def filter_pose(self, d):
        """:250-271"""
        visible = d['visible']
        q = G.angle_axis_to_quaternion(d['smpl_orient_cam'].float())
        jump = G.quat_angle_diff(q[1:], q[:-1])
        ind = (torch.where((jump > np.pi / 3) & visible[1:].bool())[0] + 1).tolist()
        for i in ind:
            if visible[i - 1]:
                if i + 1 < q.shape[0] and visible[i + 1] and (i + 1) not in ind:
                    visible[i - 1] = 0
                else:
                    visible[i] = 0
        if self.flag_make_invis_with_keypoint:
            vis_ind = torch.where(visible == 1.0)[0]
            nvalid = (d['kp_2d_score'][vis_ind] > self.make_invis_keypoint_min_score).sum(dim=1)
            visible[vis_ind[nvalid < self.make_invis_keypoint_min_num]] = 0.0
        d['vis_frames'] = visible == 1
        d['invis_frames'] = visible == 0

    def infer_motion_traj(self, d):
        """:353-392"""
        if self.mt_model is None:
            return
        ex = d['exist_frames']
        batch = {'in_body_pose': d['smpl_pose_nofill'][ex].unsqueeze(0).clone(), 'frame_mask': d['visible'][ex].unsqueeze(0).clone()}
        out = self.mt_model.inference(batch, sample_num=1)
        self._take_prior_output(d, out, 0)

    def infer_motion_traj_all(self, persons):
        """The reference runs the learned prior once per person with batch size 1 (:230-232 -> :353-392).  When every
        person exists for the same number of frames and the prior object declares `supports_person_batch`, the persons
        form one batch [P, T, 69] instead (SURVEY.md §8(f)-1): same per-person arithmetic, P times fewer launches."""
        if self.mt_model is None:
            return
        ds = list(persons.values())
        lens = {int(d['exist_len']) for d in ds}
        if len(ds) > 1 and len(lens) == 1 and getattr(self.mt_model, 'supports_person_batch', False):
            batch = {'in_body_pose': torch.stack([d['smpl_pose_nofill'][d['exist_frames']] for d in ds]),
                     'frame_mask': torch.stack([d['visible'][d['exist_frames']] for d in ds])}
            out = self.mt_model.inference(batch, sample_num=1)
            for b, d in enumerate(ds):
                self._take_prior_output(d, out, b)
        else:
            for d in ds:
                self.infer_motion_traj(d)

    def _take_prior_output(self, d, out, b):
        """:368-392 for batch row b of the prior's output"""
        ex = d['exist_frames']
        if self.flag_infill_motion:
            d['infilled'] = True
            d['smpl_pose'] = d['smpl_pose'].detach().clone()
            d['smpl_pose'][ex] = out['infer_out_body_pose'][b, 0].to(d['smpl_pose'])
        if self.flag_pred_traj:
            d['traj_predicted'] = True
            d['traj_local_pred'] = out['infer_out_local_traj_tp'][:, b, 0, :].clone().float()
            d['smpl_orient_world_base'] = d['smpl_orient_world_base'].detach().clone()
            d['root_trans_world_base'] = d['root_trans_world_base'].detach().clone()
            if 'infer_out_pose' in out:
                d['smpl_orient_world_base'][ex] = out['infer_out_pose'][b, 0, :, :3].to(d['smpl_orient_world_base'])
            if 'infer_out_orient' in out:
                d['smpl_orient_world_base'][ex] = out['infer_out_orient'][b, 0].to(d['smpl_orient_world_base'])
            d['root_trans_world_base'][ex] = out['infer_out_trans'][b, 0].to(d['root_trans_world_base'])
            d['smpl_orient_world'] = d['smpl_orient_world_base']
            d['root_trans_world'] = d['root_trans_world_base']

    def init_default_traj(self, d):
        """:319-323"""
        d['root_trans_world_base'][:] = torch.tensor([0.0, 0.0, 0.8], device=self.device)
        d['smpl_orient_world_base'][:] = G.quaternion_to_angle_axis(torch.tensor([[0.0, 0.0, 0.7071, 0.7071]], device=self.device))[0]
        d['root_trans_world'] = d['root_trans_world_base']
        d['smpl_orient_world'] = d['smpl_orient_world_base']

    def init_cam_pose(self, data, all_frames=False):
        """:294-317"""
        cands = [torch.matmul(d['person_transform_world'], d['person2cam']) * d['vis_frames'][:, None, None]
                 for d in data['person_data'].values()]
        npers = data['fr_num_persons']
        has = npers > 0
        start = torch.where(has)[0][0]
        inv = torch.zeros_like(data['cam_pose'])
        inv[has] = cands[0][has]
        data['pose_infer_cam_pose_inv'] = inv
        if all_frames:
            if not torch.all(has):
                last = inv[start]
                for i in range(len(npers)):
                    if npers[i] == 0:
                        data['cam_pose_inv'][i] = last
                    else:
                        last = data['cam_pose_inv'][i]
        else:
            inv[...] = inv[start].clone()
        inv[:, :3, :3] = G.rot6d_to_rotmat(G.rotmat_to_rot6d(inv[:, :3, :3]))
        data['cam_pose_inv'] = inv
        data['cam_pose'] = G.inverse_transform(inv)

    def _traj_local2global(self, local, local_heading=True):
        """traj_pred/utils/traj_utils.py:65-88 for one sequence [T,11] -> trans [T,3], orient_q [T,4]"""
        T = local.shape[0]
        loc = local.reshape(T, 1, 11).contiguous().float()
        trans = torch.empty((T, 1, 3), device=self.device)
        oq = torch.empty((T, 1, 4), device=self.device)
        scratch = torch.empty(T * 3, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self._lib.glamr_traj_local2global(T, 1, L.ptr(loc), int(local_heading), L.ptr(trans), L.ptr(oq), L.ptr(scratch),
                                                      L.stream_ptr()), 'glamr_traj_local2global')
        return trans[:, 0], oq[:, 0]

    def _traj_global2local(self, trans, orient_q):
        """traj_pred/utils/traj_utils.py:44-62 (init only)"""
        base = torch.tensor([0.5, 0.5, 0.5, 0.5], device=self.device)
        xy, z = trans[..., :2], trans[..., 2]
        q = G.quat_mul(orient_q, G.quat_conjugate(base).expand_as(orient_q))
        heading = G.get_heading(q)
        d6 = G.quat_to_rot6d(G.deheading_quat(q, G.get_heading_q(q)))
        d_heading = torch.cat([heading[:1], heading[1:] - heading[:-1]])
        hvec = G.heading_to_vec(d_heading)
        dxy = xy[1:] - xy[:-1]
        th = -heading[:-1]
        c, s = torch.cos(th), torch.sin(th)
        dxy_h = torch.stack([dxy[:, 0] * c - dxy[:, 1] * s, dxy[:, 0] * s + dxy[:, 1] * c], dim=-1)
        return torch.cat([torch.cat([xy[:1], dxy_h]), z.unsqueeze(-1), d6, hvec], dim=-1)

    def _interp_orient_q_sep_heading(self, orient_q_vis, vis_frames):
        """traj_pred/utils/traj_utils.py:120-142 (SciPy linear interpolation on the host, as the reference)"""
        base = torch.tensor([0.5, 0.5, 0.5, 0.5], device=self.device)
        q = G.quat_mul(orient_q_vis, G.quat_conjugate(base).expand_as(orient_q_vis))
        hq = G.get_heading_q(q)
        hvec = G.heading_to_vec(G.get_heading(q))
        d6 = G.quat_to_rot6d(G.deheading_quat(q, hq))
        n = vis_frames.shape[0]
        if int(vis_frames.sum()) == n:
            hvec_i, d6_i = hvec, d6             # every frame is a sample point: linear interpolation returns the samples
        else:
            packed = torch.cat([hvec, d6], dim=-1).cpu().numpy()          # one device->host copy for both interpolants
            vis_ind = np.where(vis_frames.cpu().numpy())[0]
            f = interp1d(vis_ind, packed, axis=0, assume_sorted=True, fill_value='extrapolate')
            both = torch.tensor(f(np.arange(n, dtype=np.float32)), device=self.device, dtype=torch.float32)
            hvec_i, d6_i = both[:, :2].contiguous(), both[:, 2:].contiguous()
        out = G.quat_mul(G.heading_to_quat(G.vec_to_heading(hvec_i)), G.rot6d_to_quat(d6_i))
        return G.quat_mul(out, base.expand_as(out))

    def init_traj_heading_from_cam(self, data):
        """:273-292"""
        for d in data['person_data'].values():
            world = torch.matmul(data['cam_pose_inv'], d['person_transform_cam'])
            q = G.rotation_matrix_to_quaternion(world[:, :3, :3].contiguous())
            q_interp = self._interp_orient_q_sep_heading(q[d['vis_frames']], d['vis_frames'])
            local = self._traj_global2local(world[:, :3, 3], q_interp)
            for (s, e) in self.cam_fix_frames:
                d['traj_local_pred'][s:e, -2:] = local[d['exist_frames']][s:e, -2:]
            trans, oq = self._traj_local2global(d['traj_local_pred'])
            ex = d['exist_frames']
            d['smpl_orient_world_base'] = d['smpl_orient_world_base'].detach().clone()
            d['root_trans_world_base'] = d['root_trans_world_base'].detach().clone()
            d['smpl_orient_world_base'][ex] = G.quaternion_to_angle_axis(oq)
            d['root_trans_world_base'][ex] = trans
            d['smpl_orient_world'] = d['smpl_orient_world_base'].clone()
            d['root_trans_world'] = d['root_trans_world_base'].clone()
            d['person_transform_world'] = G.make_transform(d['smpl_orient_world'], d['root_trans_world'], 'axis_angle')

    def init_data(self, in_dict):
        if self.est_type != 'hybrik':
            raise ValueError(f'est_type {self.est_type} not supported')
        dev = self.device
        num_fr = len(in_dict['est'][0]['bboxes_dict']['exist'])
        cam_pose = torch.eye(4, device=dev).repeat(num_fr, 1, 1)
        cam_pose_inv = G.inverse_transform(cam_pose)
        persons = {}
        for idx, est in in_dict['est'].items():
            d = self._person_from_estimate(est, in_dict['gt'].get(idx))
            if self.flag_filter_pose:
                self.filter_pose(d)
            d['root_trans_world'] = G.transform_trans(cam_pose_inv, d['root_trans_cam'].float())
            d['smpl_orient_world'] = G.transform_rot(cam_pose_inv, d['smpl_orient_cam'].float())
            d['root_trans_world_base'] = d['root_trans_world'].clone()
            d['smpl_orient_world_base'] = d['smpl_orient_world'].clone()
            d['smpl_pose_nofill'] = d['smpl_pose'].clone()
            d['smpl_pose_nofill'][~d['exist_frames']] = 0.0
            persons[idx] = d
        if self.flag_infer_motion_traj:
            self.infer_motion_traj_all(persons)
        if not (self.flag_infer_motion_traj and self.flag_pred_traj):
            raise NotImplementedError('flag_pred_traj=false (default trajectory) is not implemented in the CUDA path')
        for d in persons.values():
            d['person_transform_world'] = G.make_transform(d['smpl_orient_world'], d['root_trans_world'], 'axis_angle')
            d['person_transform_cam'] = G.make_transform(d['smpl_orient_cam'].float(), d['root_trans_cam'].float(), 'axis_angle')
            d['person2cam'] = G.inverse_transform(d['person_transform_cam'])
        last = d
        for d in persons.values():
            if self.flag_opt_person2cam_rot or self.flag_opt_person2cam_trans:         # :173-175, all T frames
                d['person2cam_res_rot'] = torch.tensor([1., 0., 0., 0., 1., 0.], device=dev).repeat(num_fr, 1)
                d['person2cam_res_trans'] = torch.zeros(num_fr, 3, device=dev)
            d['smpl_orient_world_res'] = torch.zeros_like(last['smpl_orient_world'])
            d['root_trans_world_res'] = torch.zeros_like(last['root_trans_world'])
        rel = {}
        ids = list(persons.keys())
        for i in range(len(ids)):
            for j in range(len(ids)):
                if i != j:
                    rel[(i, j)] = torch.matmul(G.inverse_transform(persons[ids[i]]['person_transform_cam']), persons[ids[j]]['person_transform_cam'])
        for d in persons.values():
            Ln = int(d['exist_len'].sum())
            d['traj_local_xy'] = torch.zeros(2, device=dev)
            d['traj_local_dxy'] = torch.zeros(Ln - 1, 2, device=dev)
            d['traj_local_heading'] = torch.zeros(1, device=dev)
            d['traj_local_dheading'] = torch.zeros(Ln - 1, device=dev)
            d['traj_local_z'] = torch.zeros(Ln, device=dev)
            d['traj_local_rot'] = torch.zeros(Ln, 6, device=dev)
        fr_num_persons = sum(d['vis_frames'] for d in persons.values())
        n_empty = int((fr_num_persons == 0).sum())
        data = {
            'seq_name': in_dict['seq_name'], 'person_data': persons, 'seq_len': num_fr, 'fr_num_persons': fr_num_persons,
            'cam_pose': cam_pose, 'cam_pose_inv': cam_pose_inv,
            'cam_inv_rot_residual': torch.zeros(n_empty, 6, device=dev),
            'cam_inv_trans_residual': torch.zeros(num_fr if self.flag_cam_inv_trans_res_all else n_empty, 3, device=dev),
            'rel_transform_cam': rel, 'gt': in_dict['gt'], 'gt_meta': in_dict['gt_meta'],
            'meta': {'algo': 'global_recon', 'mt_cfg': getattr(self.mt_cfg, 'yml_dict', None), 'num_fr': num_fr},
        }
        self.init_cam_pose(data)
        self.init_traj_heading_from_cam(data)
        if self.flag_init_cam_all_frames:
            self.init_cam_pose(data, all_frames=True)
        self._attach(data)
        self.forward(data, [], {'stage': 'init'})
        return data

    # ------------------------------------------------------------------------------------------------ device state
    def _attach(self, data):
        """Pack the optimisation variables into theta and build the constant tables.  The CUDA handle (scratch arena,
        Adam moments, captured iteration graph) is kept across calls while (P, T, J, n_params) stay the same."""
        self._fresh_attach = True
        self._data = data
        self._layout = PB.make_layout(data, self._flags)
        self._theta = torch.zeros(self._layout.n_params, device=self.device)
        PB.bind_variables(data, self._layout, self._theta)
        self._comp = PB.StageCompiler(data, self._layout, self._flags, self.device, G.angle_axis_to_rot6d, num_joints=self.smpl.num_joints,
                                      aa_to_quat=G.angle_axis_to_quaternion)
        self._reduce = torch.zeros(self._layout.n_params + NUM_TERMS, device=self.device)
        self._terms = torch.zeros(NUM_TERMS + 1, device=self.device)
        self._stage_key = None
        # multi-GPU: contiguous shards of the frame-persons n = p*T + t (SMPL + per-frame residuals are independent per
        # frame-person, so a person may straddle two ranks; P persons on P GPUs gives one person each)
        N = self._comp.P * self._comp.T
        self._n_range = (N * self.rank // self.world, N * (self.rank + 1) // self.world)

    def _release(self, at_exit=False):
        if getattr(self, '_opt', None):
            if not at_exit:
                self._drop_peers()
            self._lib.glamr_opt_destroy(self._opt)
        self._opt = None

    # ------------------------------------------------------------------------------------------------ multi-GPU
    def _setup_peers(self):
        """Exchange CUDA-IPC handles of one small buffer per rank so that the per-iteration gradient reduction runs over
        NVLink peer memory inside the Adam kernel (include/glamr_b200.h, glamr_opt_set_peers).  Collective: every rank
        calls it at the same point.  Opt-in (GLAMR_ALLREDUCE=peer): measured on B200s it is slower than the NCCL
        all-reduce captured in the iteration graph (2 GPUs 0.167 vs 0.162 ms, 4 GPUs 0.207 vs 0.173 ms per iteration),
        so NCCL stays the default; any rank failing to map a peer also falls back to NCCL."""
        import os
        self._peer_ok, self._peer_own, self._peer_opened = False, None, []
        if self.world <= 1:
            return
        dist, lib = torch.distributed, self._lib
        want = os.environ.get('GLAMR_ALLREDUCE', 'nccl') == 'peer' and self.world <= 8
        own, handle = ctypes.c_void_p(), (ctypes.c_ubyte * 64)()
        ok = want
        if ok:
            lib.glamr_opt_peer_bytes.restype = ctypes.c_size_t
            ok = lib.glamr_peer_alloc(ctypes.c_size_t(lib.glamr_opt_peer_bytes(self._opt)), ctypes.byref(own), handle) == 0
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle) if ok else None)
        ptrs = []
        if all(h is not None for h in handles):
            for r, h in enumerate(handles):
                if r == self.rank:
                    ptrs.append(own.value)
                    continue
                p = ctypes.c_void_p()
                if lib.glamr_peer_open((ctypes.c_ubyte * 64).from_buffer_copy(h), ctypes.byref(p)) != 0:
                    ok = False
                    break
                ptrs.append(p.value)
                self._peer_opened.append(p)
        else:
            ok = False
        flag = torch.tensor([1 if ok else 0], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        self._peer_own = own if own.value else None
        if int(flag[0]) == 1:
            table = (ctypes.c_void_p * self.world)(*ptrs)
            L.check(lib.glamr_opt_set_peers(self._opt, self.rank, self.world, table), 'glamr_opt_set_peers')
            self._peer_ok = True
        else:
            self._drop_peers(collective=False)
            if self.log is not None and want:
                self.log.info('peer-memory gradient reduction unavailable; using the NCCL all-reduce')

    def _drop_peers(self, collective=True):
        lib = self._lib
        if getattr(self, '_peer_ok', False):
            torch.cuda.synchronize(self.device)
            if collective:
                torch.distributed.barrier()             # nobody may still be reading this rank's buffer
            lib.glamr_opt_set_peers(self._opt, 0, 0, None)
        for p in getattr(self, '_peer_opened', []):
            lib.glamr_peer_close(p)
        if getattr(self, '_peer_own', None) is not None:
            lib.glamr_peer_free(self._peer_own)
        self._peer_ok, self._peer_own, self._peer_opened = False, None, []

    def __del__(self):
        try:
            self._release(at_exit=True)            # no collectives in a finaliser; peer buffers die with the process
        except Exception:
            pass

    def _set_stage(self, data, opt_variables, loss_cfg, stage, reset_adam, begin=False):
        if begin:            # get_parameter side effects happen once per optimize_main, not on every forward
            PB.begin_stage_variables(data, self._layout, self._theta, self._flags, opt_variables)
        pb = self._comp.compile(self._theta, opt_variables, loss_cfg, stage, n_begin=self._n_range[0], n_end=self._n_range[1],
                                owner=(self.rank == 0))
        self._pb = pb
        dims = (pb.P, pb.T, pb.J, pb.n_params)
        if self._opt is not None and dims != getattr(self, '_opt_dims', None):
            self._release()
        with torch.cuda.device(self.device):
            if self._opt is None:
                self._opt = ctypes.c_void_p()
                L.check(self._lib.glamr_opt_create(ctypes.byref(self._opt), self.smpl.handle, ctypes.byref(pb)), 'glamr_opt_create')
                self._opt_dims = dims
                self._setup_peers()
            else:                                   # bit 1: a new sequence re-uses the handle -> scratch back to its initial zeros
                flags = int(bool(reset_adam)) | (2 if self._fresh_attach else 0)
                L.check(self._lib.glamr_opt_set_problem(self._opt, ctypes.byref(pb), flags, L.stream_ptr()), 'glamr_opt_set_problem')
        self._fresh_attach = False

    def _backward(self, for_apply=False):
        """for_apply: glamr_opt_apply follows on this stream (the optimisation loop); the library then joins its side stream there, so the
        exchange below overlaps the tail of the pipelined blend"""
        fn = self._lib.glamr_opt_backward_for_apply if for_apply else self._lib.glamr_opt_backward
        L.check(fn(self._opt, L.ptr(self._theta), L.ptr(self._reduce), L.stream_ptr()), 'glamr_opt_backward')
        if self.world > 1:                                     # the one collective of the path: packed gradient + term sums
            if getattr(self, '_peer_ok', False):              # one-shot NVLink all-reduce of the library (no NCCL call)
                L.check(self._lib.glamr_allreduce_inplace(self._opt, L.ptr(self._reduce), self._reduce.numel(), L.stream_ptr()), 'glamr_allreduce_inplace')
            else:
                torch.distributed.all_reduce(self._reduce)

    def launches_per_iteration(self):
        """kernels of the CUDA library launched per optimiser iteration for the current stage (excludes the NCCL kernel)"""
        return int(self._lib.glamr_opt_launch_count(self._opt))

    def _read(self, what, *shape):
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        L.check(self._lib.glamr_opt_read(self._opt, what, ctypes.byref(p), ctypes.byref(n)), 'glamr_opt_read')
        return _device_view(p.value, n.value, self.device).view(*shape).clone()

    def _scatter_outputs(self, data):
        """copy what forward() stores into the data dict in the reference (:421-528)"""
        P, T, J = self._comp.P, self._comp.T, self._comp.J
        ow, tw = self._read(L.R_ORIENT_WORLD, P, T, 3), self._read(L.R_TRANS_WORLD, P, T, 3)
        ob, tb = self._read(L.R_ORIENT_BASE, P, T, 3), self._read(L.R_TRANS_BASE, P, T, 3)
        kp = self._read(L.R_KP_PRED, P, T, J, 2)
        ociw, tciw = self._read(L.R_ORIENT_CIW, P, T, 3), self._read(L.R_TRANS_CIW, P, T, 3)
        tl = self._read(L.R_TRAJ_LOCAL, P, T, 11)
        jw = self._read(L.R_JOINTS_WORLD, P, T, J, 3)
        if self.world > 1:
            # per-frame-person outputs exist only on the rank that evaluated that frame-person: keep the own shard, sum over ranks
            own = torch.zeros(P * T, device=self.device)
            own[self._n_range[0]:self._n_range[1]] = 1.0
            own = own.view(P, T)
            packed = torch.cat([(x * own.view(P, T, *([1] * (x.dim() - 2)))).reshape(P * T, -1) for x in (kp, ociw, tciw, jw)], dim=1).contiguous()
            torch.distributed.all_reduce(packed)
            o = 0
            outs = []
            for x in (kp, ociw, tciw, jw):
                w = x[0, 0].numel()
                outs.append(packed[:, o:o + w].reshape(x.shape))
                o += w
            kp, ociw, tciw, jw = outs
        data['cam_pose'] = G.from34(self._read(L.R_CAM_POSE, T, 12))
        data['cam_pose_inv'] = G.from34(self._read(L.R_CAM_POSE_INV, T, 12))
        for p, d in enumerate(data['person_data'].values()):
            d['smpl_orient_world'], d['root_trans_world'] = ow[p], tw[p]
            d['smpl_orient_world_base'], d['root_trans_world_base'] = ob[p], tb[p]
            d['kp_2d_pred'] = kp[p]
            d['smpl_orient_cam_in_world'], d['root_trans_cam_in_world'] = ociw[p], tciw[p]
            d['traj_local'] = tl[p][d['exist_frames']]
            d['joints_world'] = jw[p]
            d['person_transform_world'] = G.make_transform(ow[p], tw[p], 'axis_angle')

    # ------------------------------------------------------------------------------------------------ reference API
    def forward(self, data, opt_variables, opt_meta):
        """:428-531 -- evaluates the current variables and refreshes the derived entries of `data`."""
        with torch.cuda.device(self.device):
            self._set_stage(data, opt_variables, getattr(self, '_loss_cfg', {}) or {}, opt_meta['stage'], reset_adam=False)
            self._backward()
            self._scatter_outputs(data)

    def compute_loss(self, data, loss_cfg):
        """:533-545 -> (total, weighted dict, unweighted dict) of 0-d CUDA tensors"""
        with torch.cuda.device(self.device):
            stage = getattr(self, '_cur_stage', 'opt')
            self._set_stage(data, getattr(self, '_cur_vars', []), loss_cfg, stage, reset_adam=False)
            self._backward()
            L.check(self._lib.glamr_opt_losses(self._opt, L.ptr(self._reduce), L.ptr(self._terms), L.stream_ptr()), 'glamr_opt_losses')
            terms = self._terms.clone()
        uw = {name: terms[L.TERM_INDEX[name]] for name in loss_cfg}
        wt = {name: uw[name] * loss_cfg[name]['weight'] for name in loss_cfg}
        return terms[NUM_TERMS], wt, uw

    def optimize_main(self, data, opt_variables, opt_lr, opt_niters, loss_cfg, opt_meta):
        """:547-570 -- opt_niters fused iterations (forward + residuals + backward [+ allreduce] + Adam)."""
        stage = opt_meta['stage']
        self._cur_vars, self._cur_stage, self._loss_cfg = opt_variables, stage, loss_cfg
        lib = self._lib
        with torch.cuda.device(self.device):
            self._set_stage(data, opt_variables, loss_cfg, stage, reset_adam=True, begin=True)
            hist = torch.zeros((max(opt_niters, 1), NUM_TERMS + 1), device=self.device)
            stream = torch.cuda.current_stream()

            def one_iteration():
                self._backward(for_apply=True)
                L.check(lib.glamr_opt_apply(self._opt, L.ptr(self._theta), L.ptr(self._reduce), float(opt_lr), L.ptr(hist), NUM_TERMS + 1,
                                            L.stream_ptr()), 'glamr_opt_apply')
            graph = None
            done = 0
            t_stage = time.time()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            # the library owns the loop when nothing has to happen between backward and apply: one GPU, or the reduction
            # fused into the Adam kernel over peer memory
            native = self.world == 1 or getattr(self, '_peer_ok', False)
            if native and opt_niters > 0:
                L.check(lib.glamr_opt_iterate(self._opt, L.ptr(self._theta), L.ptr(self._reduce), float(opt_lr), L.ptr(hist), NUM_TERMS + 1,
                                              1, int(self.use_cuda_graph), L.stream_ptr()), 'glamr_opt_iterate')
                done = 1
            elif opt_niters > 0:
                one_iteration()                                  # warm-up (also sets kernel attributes) = iteration 0
                done = 1
                if self.use_cuda_graph and opt_niters > 2:
                    try:                                         # the NCCL all-reduce is capturable too
                        graph = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(graph):
                            one_iteration()
                    except Exception as e:                       # capture is an optimisation, eager launches are equivalent
                        graph = None
                        torch.cuda.synchronize()
                        if self.log is not None:
                            self.log.info(f'CUDA-graph capture with NCCL unavailable ({e}); running eager iterations')
            ev0.record()
            chunk = max(int(self.log_interval), 1)
            logging_on = self.log is not None or self.specs.get('print_logs', False)
            if native and not logging_on:
                chunk = max(opt_niters, 1)
            logged = 0
            while done < opt_niters:
                todo = min(chunk, opt_niters - done)
                if native:
                    L.check(lib.glamr_opt_iterate(self._opt, L.ptr(self._theta), L.ptr(self._reduce), float(opt_lr), L.ptr(hist), NUM_TERMS + 1,
                                                  todo, int(self.use_cuda_graph), L.stream_ptr()), 'glamr_opt_iterate')
                else:
                    for _ in range(todo):
                        if graph is not None:
                            graph.replay()
                        else:
                            one_iteration()
                done += todo
                if logging_on:
                    logged = self._write_logs(hist, logged, done, opt_niters, opt_lr, loss_cfg, stage, data['seq_name'], t_stage)
            ev1.record()
            ev1.synchronize()
            if opt_niters > 1:
                self.iter_ms.append((stage, opt_niters - 1, ev0.elapsed_time(ev1) / (opt_niters - 1)))
            if self.log is not None or self.specs.get('print_logs', False):
                self._write_logs(hist, logged, done, opt_niters, opt_lr, loss_cfg, stage, data['seq_name'], t_stage)
            self.loss_history = hist
            self.cur_iter = max(opt_niters - 1, 0)
            if opt_niters > 0:
                self._scatter_outputs(data)                      # state of the last closure, like the reference
        return data

    def _write_logs(self, hist, start, end, opt_niters, opt_lr, loss_cfg, stage, seq_name, t_stage):
        """:646-659 same line format; values are read back in blocks of `log_interval` iterations."""
        if end <= start:
            return end
        vals = hist[start:end].cpu().numpy()
        per_iter = (time.time() - t_stage) / max(end, 1)
        for k, it in enumerate(range(start, end)):
            loss_str = ' | '.join(f'{name}: {vals[k, L.TERM_INDEX[name]]:7.3f}' for name in loss_cfg)
            eta = _sec_to_time(per_iter * (opt_niters - it - 1))
            info = f'{self.cfg.id} - {seq_name} - {stage} | {it:4d}/{opt_niters} | TE: {_sec_to_time(per_iter)} ETA: {eta} | LR: {opt_lr:.0e} | {loss_str}'
            if self.log is None:
                print(info)
            else:
                self.log.info(info)
        return end

    def optimize(self, in_dict, continue_opt=False):
        """:572-589"""
        t0 = time.perf_counter()
        if continue_opt:
            data = tensor_to(in_dict, self.device)
            self._attach(data)
        else:
            data = self.init_data(in_dict)
        t1 = time.perf_counter()
        for stage, stage_specs in self.opt_stage_specs.items():
            opt_meta = {'stage': stage, 'opt_latent_start_iter': stage_specs.get('opt_latent_start_iter', 0)}
            self.optimize_main(data, stage_specs['opt_variables'], stage_specs['opt_lr'], stage_specs['opt_niters'],
                               stage_specs['loss_cfg'], opt_meta)
            if stage_specs.get('reinitialize_cam', False):
                data['cam_pose'][:] = data['cam_pose'][[0]]
                data['cam_pose_inv'] = G.inverse_transform(data['cam_pose'])
        t2 = time.perf_counter()
        out = tensor_to_numpy(data)
        # host wall-clock of the three phases of the last call (init_data includes the learned prior; stages include the waits)
        self.phase_seconds = {'init_data': t1 - t0, 'stages': t2 - t1, 'to_numpy': time.perf_counter() - t2}
        return out


def _device_view(addr, count, device):
    """float32 tensor aliasing `count` floats of device memory at `addr` (owned by a CUDA-library handle)."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {'shape': (count,), 'typestr': '<f4', 'data': (addr, False), 'version': 2}
    return torch.as_tensor(h, device=device)
