"""Translate GLAMR's ``data`` dict + one stage's YAML specs into the flat description the CUDA library consumes
(``glamr_problem_t`` / ``glamr_person_t`` of include/glamr_b200.h).

* ``VariableLayout`` packs every optimisation variable of ``GlobalReconOptimizer.get_parameter``
  (global_recon/models/global_recon_model.py:591-633) into one vector ``theta``; the tensors stored in the data dict
  (``cam_rot_6d``, ``traj_local_xy`` ...) are views into it, so the dict always shows current values.
* ``StageCompiler`` turns ``loss_cfg`` (global_recon/models/loss_func.py semantics: min_conf, first_frame_only,
  first_frame_weight, visibility masks, normalisers) into per-frame weight arrays and scalar term tables.

Pure tensor bookkeeping, device agnostic (tests build it on the CPU for the host harness); nothing here computes
on the optimisation path.
"""
import ctypes

import numpy as np
import torch

from . import lib as L


class VariableLayout:
    def __init__(self, T, n_empty, trans_res_rows, lens, person2cam_res=False):
        """person2cam_res: also allocate person2cam_res_rot [T,6] + person2cam_res_trans [T,3] per person
        (flag_opt_person2cam_rot / _trans), after every other block so that the offsets above do not depend on it"""
        self.T, self.n_empty, self.trans_res_rows, self.lens = T, n_empty, trans_res_rows, list(lens)
        off = 0

        def take(n):
            nonlocal off
            o = off
            off += n
            return o
        self.cam_rot, self.cam_trans = take(6 * T), take(3 * T)
        self.cam_rot_fix, self.cam_trans_fix = take(6), take(3)
        self.cam_inv_rot_res, self.cam_inv_trans_res = take(6 * n_empty), take(3 * trans_res_rows)
        self.persons = []
        for Ln in self.lens:
            self.persons.append(dict(xy=take(2), heading=take(1), dxy=take(2 * (Ln - 1)), dheading=take(Ln - 1), z=take(Ln),
                                     rot=take(6 * Ln), world_dheading=take(T), orient_res=take(3 * T), trans_res=take(3 * T)))
        self.person2cam_res = person2cam_res
        if person2cam_res:
            for o in self.persons:          # the trans block directly follows the rot block (glamr_person_t.off_person2cam_res)
                o['p2c_rot'], o['p2c_trans'] = take(6 * T), take(3 * T)
        self.n_params = off

    def views(self, theta, p=None):
        """name -> view of theta with the reference's tensor shape"""
        T = self.T
        if p is None:
            v = lambda o, n, *shape: theta[o:o + n].view(*shape)
            return {'cam_rot_6d': v(self.cam_rot, 6 * T, T, 6), 'cam_trans': v(self.cam_trans, 3 * T, T, 3),
                    'cam_rot_6d_fix': v(self.cam_rot_fix, 6, 1, 6), 'cam_trans_fix': v(self.cam_trans_fix, 3, 1, 3),
                    'cam_inv_rot_residual': v(self.cam_inv_rot_res, 6 * self.n_empty, self.n_empty, 6),
                    'cam_inv_trans_residual': v(self.cam_inv_trans_res, 3 * self.trans_res_rows, self.trans_res_rows, 3)}
        o, Ln = self.persons[p], self.lens[p]
        v = lambda k, n, *shape: theta[o[k]:o[k] + n].view(*shape)
        out = {'traj_local_xy': v('xy', 2, 2), 'traj_local_heading': v('heading', 1, 1),
               'traj_local_dxy': v('dxy', 2 * (Ln - 1), Ln - 1, 2), 'traj_local_dheading': v('dheading', Ln - 1, Ln - 1),
               'traj_local_z': v('z', Ln, Ln), 'traj_local_rot': v('rot', 6 * Ln, Ln, 6),
               'world_dheading': v('world_dheading', T, T, 1), 'smpl_orient_world_res': v('orient_res', 3 * T, T, 3),
               'root_trans_world_res': v('trans_res', 3 * T, T, 3)}
        if self.person2cam_res:
            out['person2cam_res_rot'], out['person2cam_res_trans'] = v('p2c_rot', 6 * T, T, 6), v('p2c_trans', 3 * T, T, 3)
        return out


def _f32(x, device):
    return torch.as_tensor(x).to(device=device, dtype=torch.float32).contiguous()


class StageCompiler:
    """Holds the per-person constant tensors and builds a ``Problem`` for every stage."""

    def __init__(self, data, layout, flags, device, aa_to_rot6d, num_joints=26, aa_to_quat=None):
        """flags: dict with flag_fixed_cam, flag_opt_cam, flag_opt_cam_from_person_pose, flag_cam_inv_trans_res_all,
        flag_opt_vis_local_rot, cam_fix_frames and optionally flag_opt_person2cam_rot / flag_opt_person2cam_trans (default
        off).  aa_to_rot6d: callable (device math lives in the CUDA library)."""
        self.data, self.layout, self.flags, self.device, self.J = data, layout, flags, device, num_joints
        self.pids = list(data['person_data'].keys())
        self.P, self.T = len(self.pids), data['seq_len']
        T, dev = self.T, device
        self.keep = []                               # tensors whose storage the structs point into
        self.const = []
        pose_all, beta_all, scale_all = [], [], []
        for pid in self.pids:
            d = data['person_data'][pid]
            start, Ln = int(d['fr_start']), int(d['exist_len'])
            mask = torch.ones(max(Ln - 1, 0))
            for (s, e) in flags['cam_fix_frames']:
                mask[s:e] = 0.0
            c = {
                'start': start, 'len': Ln,
                'traj_local_pred': _f32(d['traj_local_pred'], dev),
                'orient_base_init': _f32(d['smpl_orient_world_base'], dev).clone(),
                'trans_base_init': _f32(d['root_trans_world_base'], dev).clone(),
                'cam_K': _f32(d['cam_K'], dev).reshape(T, 9),
                'kp_target': _f32(d['kp_2d_aligned'], dev),
                'orient_cam_6d': _f32(aa_to_rot6d(_f32(d['smpl_orient_cam'], dev)), dev),
                'orient_cam_q': None if aa_to_quat is None else _f32(aa_to_quat(_f32(d['smpl_orient_cam'], dev)), dev),
                'trans_cam': _f32(d['root_trans_cam'], dev),
                'person2cam': _f32(d['person2cam'], dev)[:, :3, :].reshape(T, 12).contiguous(),
                'dheading_mask': _f32(mask, dev),
                'rot_mask': _f32(d['vis_frames'][start:start + Ln], dev) if flags.get('flag_opt_vis_local_rot', False) else None,
                'vis': _f32(d['vis_frames'], dev),
            }
            self.const.append(c)
            pose_all.append(_f32(d['smpl_pose'], dev))
            beta_all.append(_f32(d['smpl_beta'], dev))
            scale_all.append(None if d['scale'] is None else _f32(d['scale'], dev))
        self.pose_all = torch.stack(pose_all).contiguous()
        self.beta_all = torch.stack(beta_all).contiguous()
        self.scale_all = None if scale_all[0] is None else torch.stack(scale_all).contiguous()
        # host copies of what the per-stage weight tables are built from (visibility, keypoint scores, persons per frame):
        # ONE device->host copy here instead of several per person and stage
        P_, J_ = self.P, self.J
        packed = torch.cat([torch.stack([torch.as_tensor(data['person_data'][pid]['vis_frames']).to(dev).double() for pid in self.pids]).reshape(-1),
                            torch.stack([torch.as_tensor(data['person_data'][pid]['kp_2d_score']).to(dev).double() for pid in self.pids]).reshape(-1),
                            torch.as_tensor(data['fr_num_persons']).to(dev).double().reshape(-1)]).cpu()
        self.host_vis = packed[:P_ * T].reshape(P_, T) > 0.5
        self.host_score = packed[P_ * T:P_ * T + P_ * T * J_].reshape(P_, T, J_)
        # camera-from-persons bookkeeping (global_recon_model.py:489-506)
        npers = packed[P_ * T + P_ * T * J_:].to(torch.int64)
        has = npers > 0
        first = int(torch.where(has)[0][0])
        src, empty_idx, last, ne = [], [], first, 0
        for t in range(T):
            if npers[t] > 0:
                last = t
                empty_idx.append(-1)
            else:
                empty_idx.append(ne)
                ne += 1
            src.append(last)
        self.fill_src = torch.tensor(src, dtype=torch.int32, device=dev)
        self.empty_index = torch.tensor(empty_idx, dtype=torch.int32, device=dev)
        self.inv_num = _f32(torch.where(has, 1.0 / npers.clamp(min=1).float(), torch.zeros(T)), dev)
        rel = data.get('rel_transform_cam')
        if rel:
            tgt = torch.zeros(self.P * self.P, T, 12, device=dev)
            for (i, j), C in rel.items():
                tgt[i * self.P + j] = torch.as_tensor(C).detach().to(dev).float()[:, :3, :].reshape(T, 12)
            self.rel_target = tgt.contiguous()
        else:
            self.rel_target = None

    # ------------------------------------------------------------------------------------------------ per stage
    def _person_weights(self, p, loss_cfg):
        T, J = self.T, self.J
        vis, score = self.host_vis[p], self.host_score[p]
        vis_idx = torch.where(vis)[0]
        nvis = int(vis.sum())
        kp_w, kp_dm = torch.zeros(T, J, dtype=torch.float64), torch.zeros(T, J, dtype=torch.float64)
        ctr_w, ctt_w = torch.zeros(T, dtype=torch.float64), torch.zeros(T, dtype=torch.float64)
        norms = {}
        if 'kp_2d' in loss_cfg:                                              # loss_func.py:15-36
            sp = loss_cfg['kp_2d']
            conf = score.clone()
            conf[conf < sp.get('min_conf', 0.05)] = 0
            ffw = sp.get('first_frame_weight', 1.0)
            if sp.get('first_frame_only', False):
                kp_w[vis_idx[0]] = ffw * (conf[vis] ** 2).sum(0)           # rho of frame 0 broadcast over all frames' scores
            else:
                fw = torch.ones(nvis, dtype=torch.float64)
                fw[:10] = ffw
                kp_w[vis] = conf[vis] ** 2 * fw[:, None]
            norms['kp_2d'] = nvis
        if 'kp_2d_dist' in loss_cfg:                                         # loss_func.py:39-57
            sp = loss_cfg['kp_2d_dist']
            m = (score > sp.get('min_conf', 0.05)).double()
            if sp.get('first_frame_only', False):
                m[1:] = 0
            kp_dm = m
            norms['kp_2d_dist'] = float(m.sum())
        if 'cam_traj_rot' in loss_cfg:                                       # loss_func.py:147-172
            sp = loss_cfg['cam_traj_rot']
            if sp.get('rot_type', '6d') not in ('6d', 'quat'):
                raise ValueError(f"cam_traj_rot: unknown rot_type {sp.get('rot_type')}")
            if sp.get('first_frame_only', False):
                ctr_w[vis_idx[0]] = 1.0
                norms['cam_traj_rot'] = 1
            else:
                ctr_w[vis] = 1.0
                ctr_w[vis_idx[0]] = sp.get('first_frame_weight', 1.0) ** 2
                norms['cam_traj_rot'] = nvis
        if 'cam_traj_trans' in loss_cfg:                                     # loss_func.py:175-186
            sp = loss_cfg['cam_traj_trans']
            ctt_w[vis] = 1.0
            ctt_w[vis_idx[0]] = sp.get('first_frame_weight', 1.0) ** 2
            norms['cam_traj_trans'] = nvis
        return kp_w, kp_dm, ctr_w, ctt_w, norms

    def compile(self, theta, opt_variables, loss_cfg, stage, n_begin=0, n_end=None, owner=True):
        data, lay, fl, dev, P, T, J = self.data, self.layout, self.flags, self.device, self.P, self.T, self.J
        n_end = P * T if n_end is None else n_end
        for name in loss_cfg:
            if name == 'person2cam_res_trans_reg':
                raise NotImplementedError(
                    "residual 'person2cam_res_trans_reg' fails in the reference itself (loss_func.py:244-245 looks up "
                    "'person2cam_res_trans' in the top-level data dict, but the variable lives in each person's dict: KeyError), "
                    "so it has no semantics to match")
            if name not in L.TERM_INDEX:
                raise NotImplementedError(f"residual '{name}' has no CUDA implementation (no CPU fallback)")
        pb = L.Problem()
        pb.P, pb.T, pb.J, pb.n_params = P, T, J, lay.n_params
        pb.n_begin, pb.n_end, pb.owner = n_begin, n_end, int(owner)
        keep = []
        # ---- camera mode (global_recon_model.py:473-508)
        mode = L.CAM_CONST
        if fl['flag_opt_cam'] and stage != 'init':
            if 'cam' in opt_variables:
                mode = L.CAM_FIXED if fl['flag_fixed_cam'] else L.CAM_PER_FRAME
            elif fl['flag_opt_cam_from_person_pose']:
                mode = L.CAM_FROM_PERSONS
        pb.cam_mode = mode
        if mode == L.CAM_FIXED:
            pb.off_cam_rot, pb.off_cam_trans = lay.cam_rot_fix, lay.cam_trans_fix
        elif mode == L.CAM_PER_FRAME:
            pb.off_cam_rot, pb.off_cam_trans = lay.cam_rot, lay.cam_trans
        else:
            pb.off_cam_rot, pb.off_cam_trans = lay.cam_inv_rot_res, lay.cam_inv_trans_res
        cam_const = _f32(data['cam_pose'], dev)[:, :3, :].reshape(T, 12).contiguous().clone()
        keep.append(cam_const)
        pb.cam_pose_const = cam_const.data_ptr()
        pb.trans_res_all = int(fl['flag_cam_inv_trans_res_all'])
        pb.use_world_res = int('world_res' in opt_variables)
        pb.has_world_dheading = int(any('world_dheading' in data['person_data'][pid] for pid in self.pids))
        pb.empty_index, pb.fill_src, pb.inv_num_persons = self.empty_index.data_ptr(), self.fill_src.data_ptr(), self.inv_num.data_ptr()
        pb.smpl_pose_all, pb.smpl_beta_all = self.pose_all.data_ptr(), self.beta_all.data_ptr()
        pb.scale_all = None if self.scale_all is None else self.scale_all.data_ptr()
        # ---- persons
        persons = (L.Person * P)()
        norms = {}
        host_w = torch.zeros(P, 2 * T * J + 2 * T, dtype=torch.float32)        # [kp_w | kp_dist_mask | ctr_w | ctt_w] per person
        for p in range(P):
            kp_w, kp_dm, ctr_w, ctt_w, nrm = self._person_weights(p, loss_cfg)
            host_w[p] = torch.cat([kp_w.reshape(-1), kp_dm.reshape(-1), ctr_w, ctt_w]).float()
            for k, v in nrm.items():
                norms[k] = norms.get(k, 0) + v
        dev_w = host_w.to(dev)                                                   # one upload for all persons
        keep.append(dev_w)
        for p, pid in enumerate(self.pids):
            d, c, o = data['person_data'][pid], self.const[p], lay.persons[p]
            ps = persons[p]
            ps.start, ps.len = c['start'], c['len']
            ps.off_xy, ps.off_heading, ps.off_dxy, ps.off_dheading = o['xy'], o['heading'], o['dxy'], o['dheading']
            ps.off_z, ps.off_rot, ps.off_world_dheading = o['z'], o['rot'], o['world_dheading']
            ps.off_orient_res, ps.off_trans_res = o['orient_res'], o['trans_res']
            # composed whenever the variables exist (camera-from-persons mode only; a stage that does not optimise them
            # uses their current value)
            ps.off_person2cam_res = o['p2c_rot'] if lay.person2cam_res else -1
            for name in ['traj_local_pred', 'orient_base_init', 'trans_base_init', 'cam_K', 'kp_target', 'orient_cam_6d',
                         'orient_cam_q', 'trans_cam', 'person2cam', 'dheading_mask', 'rot_mask', 'vis']:
                setattr(ps, name, None if c[name] is None else c[name].data_ptr())
            base = dev_w.data_ptr() + p * dev_w.shape[1] * 4
            ps.kp_w, ps.kp_dist_mask = base, base + T * J * 4
            ps.ctr_w, ps.ctt_w = base + 2 * T * J * 4, base + (2 * T * J + T) * 4
        persons_dev = torch.frombuffer(bytearray(bytes(persons)), dtype=torch.uint8).to(dev)
        keep.append(persons_dev)
        pb.persons = persons_dev.data_ptr()
        # ---- rel_transform (loss_func.py:248-271)
        if self.rel_target is not None and 'rel_transform' in loss_cfg:
            sp = loss_cfg['rel_transform']
            ffw = sp.get('first_frame_weight', 10)
            rw, rwt = torch.zeros(P * P, T), torch.zeros(P * P, T)
            n_rel = 0
            for (i, j) in data['rel_transform_cam'].keys():
                n_rel += T
                both = self.host_vis[i] & self.host_vis[j]
                if both.sum() == 0:
                    continue
                f0 = int(torch.where(both)[0][0])
                wv = both.float()
                wv[f0] = float(ffw) ** 2
                rw[i * P + j] = wv
                wt = wv.clone()
                if sp.get('first_frame_trans_only', False):
                    wt[:] = 0
                    wt[f0] = float(ffw) ** 2
                rwt[i * P + j] = wt
            rw, rwt = rw.to(dev).contiguous(), rwt.to(dev).contiguous()
            keep += [rw, rwt]
            pb.rel_target, pb.rel_w, pb.rel_wt = self.rel_target.data_ptr(), rw.data_ptr(), rwt.data_ptr()
            pb.rel_trans_weight = sp.get('trans_weight', 1.0)
            norms['rel_transform'] = n_rel
        elif 'rel_transform' in loss_cfg:
            norms['rel_transform'] = 0
        # ---- scalar term tables
        lens = lay.lens
        norms.update({
            'traj_rot_smoothness': P * (T - 1), 'traj_trans_smoothness': P * (T - 1),
            'local_traj_dxy_reg': sum(n - 1 for n in lens), 'local_traj_dheading_reg': sum(n - 1 for n in lens),
            'local_traj_dheading_reg_new': sum(n - 1 for n in lens), 'local_traj_rot_reg': sum(lens), 'local_traj_z_reg': sum(lens),
            'traj_rot_res': P * T, 'traj_trans_res': P * T, 'cam_inv_trans_residual_reg': lay.trans_res_rows,
            'cam_inv_rot_smoothness': T - 1, 'cam_origin_smoothness': T - 1, 'cam_rot_smoothness': T - 1, 'cam_trans_smoothness': T - 1,
            'cam_depth_smoothness': 1,          # loss_func.py:102 sums over the T-1 frame pairs (the .mean() sees a 0-d tensor)
        })
        pb.cam_traj_rot_quat = int(loss_cfg.get('cam_traj_rot', {}).get('rot_type', '6d') == 'quat')
        pb.traj_rot_smooth_quat = int(loss_cfg.get('traj_rot_smoothness', {}).get('rot_type', '6d') == 'quat')
        if (pb.cam_traj_rot_quat or pb.traj_rot_smooth_quat) and self.const[0]['orient_cam_q'] is None:
            raise ValueError("rot_type 'quat' needs the aa_to_quat callable (StageCompiler(..., aa_to_quat=...))")
        if 'cam_up_reg' in loss_cfg:
            sp = loss_cfg['cam_up_reg']
            pb.cam_up_first_weight = sp.get('first_frame_weight', 1.0)
            pb.cam_up_first_only = int(sp.get('first_frame_only', False))
            norms['cam_up_reg'] = 1 if pb.cam_up_first_only else T
        if ('cam_rot_smoothness' in loss_cfg or 'cam_trans_smoothness' in loss_cfg) and mode != L.CAM_PER_FRAME:
            raise NotImplementedError('cam_rot/trans_smoothness need per-frame camera variables')
        for name, sp in loss_cfg.items():
            k = L.TERM_INDEX[name]
            pb.term_enabled[k] = 1
            pb.term_monitor[k] = int(sp.get('monitor_only', False))
            pb.term_weight[k] = float(sp['weight'])
            n = float(norms.get(name, 1))
            pb.term_norm[k] = n if n > 0 else 1.0
        # ---- which entries of theta Adam updates (get_parameter, :591-633)
        active = torch.zeros(lay.n_params, dtype=torch.uint8)

        def on(o, n):
            active[o:o + n] = 1
        if 'cam' not in opt_variables:
            on(lay.cam_inv_rot_res, 6 * lay.n_empty)
            on(lay.cam_inv_trans_res, 3 * lay.trans_res_rows)
        elif fl['flag_fixed_cam']:
            on(lay.cam_rot_fix, 6)
            on(lay.cam_trans_fix, 3)
        else:
            on(lay.cam_rot, 6 * T)
            on(lay.cam_trans, 3 * T)
        sizes = lambda Ln: {'xy': 2, 'heading': 1, 'dxy': 2 * (Ln - 1), 'dheading': Ln - 1, 'z': Ln, 'rot': 6 * Ln}
        for p in range(P):
            o, sz = lay.persons[p], sizes(lens[p])
            for key in opt_variables:
                if key == 'world_res':
                    on(o['orient_res'], 3 * T)
                    on(o['trans_res'], 3 * T)
                if 'local' in key:
                    name = key[len('local_'):]
                    if name not in sz:
                        raise KeyError(f'unknown optimisation variable {key}')
                    on(o[name], sz[name])
                if key == 'world_dheading':
                    on(o['world_dheading'], T)
                # listed without its flag, the reference does not optimise it (global_recon_model.py:616-619)
                if key == 'person2cam_rot' and fl.get('flag_opt_person2cam_rot', False):
                    on(o['p2c_rot'], 6 * T)
                if key == 'person2cam_trans' and fl.get('flag_opt_person2cam_trans', False):
                    on(o['p2c_trans'], 3 * T)
                if key == 'world_dxy':
                    raise NotImplementedError(f"optimisation variable '{key}' is not implemented in the CUDA path")
        active = active.to(dev)
        keep.append(active)
        pb.active = active.data_ptr()
        self.keep = keep
        return pb


# ---------------------------------------------------------------------------------------------------- variables
def make_layout(data, flags):
    persons = data['person_data']
    T = data['seq_len']
    n_empty = int((torch.as_tensor(data['fr_num_persons']) == 0).sum())
    rows = T if flags['flag_cam_inv_trans_res_all'] else n_empty
    p2c = flags.get('flag_opt_person2cam_rot', False) or flags.get('flag_opt_person2cam_trans', False)
    return VariableLayout(T, n_empty, rows, [int(d['exist_len']) for d in persons.values()], person2cam_res=p2c)


def bind_variables(data, layout, theta):
    """Move every optimisation variable that already exists in `data` into the packed vector `theta` and replace the
    dict entry by the view, so later reads (and the final tensor_to_numpy) see what the kernels update."""
    gv = layout.views(theta)
    for name in ['cam_inv_rot_residual', 'cam_inv_trans_residual']:
        gv[name].copy_(torch.as_tensor(data[name]).to(theta))
        data[name] = gv[name]
    for p, d in enumerate(data['person_data'].values()):
        pv = layout.views(theta, p)
        if layout.person2cam_res:
            # a dict without them (continue_opt from a run without the flags) starts from the initial value of
            # global_recon_model.py:173-175: identity 6d rotation, zero translation
            d.setdefault('person2cam_res_rot', torch.tensor([1., 0., 0., 0., 1., 0.]).repeat(layout.T, 1))
            d.setdefault('person2cam_res_trans', torch.zeros(layout.T, 3))
        for name in ['traj_local_xy', 'traj_local_heading', 'traj_local_dxy', 'traj_local_dheading', 'traj_local_z',
                     'traj_local_rot', 'smpl_orient_world_res', 'root_trans_world_res', 'world_dheading',
                     'person2cam_res_rot', 'person2cam_res_trans']:
            # world_dheading exists once a stage has requested it (global_recon_model.py:624-627); with continue_opt it
            # arrives already optimised and forward() keeps composing with it (:459-465)
            if name in d and name in pv:
                pv[name].copy_(torch.as_tensor(d[name]).to(theta))
                d[name] = pv[name]


def begin_stage_variables(data, layout, theta, flags, opt_variables):
    """Side effects of GlobalReconOptimizer.get_parameter (global_recon_model.py:596-631): camera variables are
    re-initialised from the current cam_pose, world_dheading is created (zeros) the first time it is requested."""
    gv = layout.views(theta)
    if 'cam' in opt_variables:
        cam = torch.as_tensor(data['cam_pose']).to(theta)
        d6 = torch.cat([cam[:, :3, 0], cam[:, :3, 1]], dim=-1)           # rotmat_to_rot6d: first two columns
        if flags['flag_fixed_cam']:
            gv['cam_rot_6d_fix'].copy_(d6[:1])
            gv['cam_trans_fix'].copy_(cam[:1, :3, 3])
            data['cam_rot_6d_fix'], data['cam_trans_fix'] = gv['cam_rot_6d_fix'], gv['cam_trans_fix']
            data['cam_rot_6d'] = gv['cam_rot_6d_fix'].expand(layout.T, -1)
            data['cam_trans'] = gv['cam_trans_fix'].expand(layout.T, -1)
        else:
            gv['cam_rot_6d'].copy_(d6)
            gv['cam_trans'].copy_(cam[:, :3, 3])
            data['cam_rot_6d'], data['cam_trans'] = gv['cam_rot_6d'], gv['cam_trans']
    if 'world_dheading' in opt_variables:
        for p, d in enumerate(data['person_data'].values()):
            if 'world_dheading' not in d:
                d['world_dheading'] = layout.views(theta, p)['world_dheading']
