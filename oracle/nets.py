"""ORACLE (test infrastructure): torch-CPU restatement of GLAMR's learned-prior INFERENCE path with the reference's
state-dict key names, so seeded weights (glamr_b200.synthetic_nets) or real checkpoints load into it unchanged.

  MotionInfiller     motion_infiller/models/motion_infiller_vae.py: ContextEncoder :22-123, DataDecoder :252-421,
                     windowed autoregressive inference :564-632 (shipped cfg motion_infiller/cfg/motion_infiller_demo.yml)
  TrajPredictor      traj_pred/models/traj_pred_vae.py: ContextEncoder :20-92, DataDecoder :202-333, inference :524-548
                     (traj_pred/cfg/traj_pred_demo.yml), with lib/models/{mlp,rnn,pos_encoding}.py and lib/utils/dist.py
  MotionTrajJoint    motion_infiller/models/motion_traj_joint_model.py:73-145 (infill -> FK joints -> trajectory)

torch.nn.TransformerEncoder/DecoderLayer, nn.LSTMCell are the same library modules the reference instantiates; what
is restated is GLAMR's wiring around them.  Training-only parts (posterior encoders, losses) are not on the path.
"""
import numpy as np
import torch
from torch import nn

from . import rotations as rt
from . import traj_codec as tc

NZ, D, PAST, CUR, FUT = 128, 256, 10, 30, 10


class _MLP(nn.Module):
    """lib/models/mlp.py:9-41 (activation after EVERY layer)"""

    def __init__(self, din, hdims):
        super().__init__()
        self.affine_layers = nn.ModuleList()
        for h in hdims:
            self.affine_layers.append(nn.Linear(din, h))
            din = h

    def forward(self, x):
        for lin in self.affine_layers:
            x = torch.relu(lin(x))
        return x


class _PosEnc(nn.Module):
    """lib/models/pos_encoding.py:6-82, enc_type 'original', concat=True"""

    def __init__(self, enc_dim, in_dim):
        super().__init__()
        self.enc_dim = enc_dim
        self.fc = nn.Linear(enc_dim + in_dim, enc_dim)

    def forward(self, x, pos_offset=0):
        pos = torch.arange(x.shape[0], device=x.device) + pos_offset
        mul = torch.exp(torch.arange(0, self.enc_dim, 2, device=x.device) * (-np.log(10000.0) / self.enc_dim))
        ang = pos.unsqueeze(-1) * mul
        pe = torch.stack([torch.sin(ang), torch.cos(ang)], dim=-1).view(-1, 1, self.enc_dim)
        return self.fc(torch.cat([x, pe.expand(x.shape[:-1] + (self.enc_dim,))], dim=-1))


class _BiLSTM(nn.Module):
    """lib/models/rnn.py:5-61: LSTMCell loops, zero initial state, outputs concatenated (forward | backward)"""

    def __init__(self, din, dout):
        super().__init__()
        self.rnn_f = nn.LSTMCell(din, dout // 2)
        self.rnn_b = nn.LSTMCell(din, dout // 2)

    def _run(self, cell, x, reverse):
        h = torch.zeros(x.shape[1], cell.hidden_size, dtype=x.dtype)
        c = torch.zeros_like(h)
        outs = [None] * x.shape[0]
        for t in (reversed(range(x.shape[0])) if reverse else range(x.shape[0])):
            h, c = cell(x[t], (h, c))
            outs[t] = h
        return torch.stack(outs, 0)

    def forward(self, x):
        return torch.cat([self._run(self.rnn_f, x, False), self._run(self.rnn_b, x, True)], dim=2)


class _InfillerContext(nn.Module):
    def __init__(self):
        super().__init__()
        self.in_fc = nn.Linear(69, D)
        self.pos_enc = _PosEnc(D, D)
        self.temporal_net = nn.TransformerEncoder(nn.TransformerEncoderLayer(D, 8, 512, 0.1), 2, enable_nested_tensor=False)


class _InfillerDecoder(nn.Module):
    def __init__(self):
        super().__init__()
        self.pos_enc = _PosEnc(D, NZ)
        self.temporal_net = nn.TransformerDecoder(nn.TransformerDecoderLayer(D, 8, 512, 0.1), 2)
        self.out_mlp = _MLP(D, [512, 256])
        self.out_fc = nn.Linear(D, 69)
        self.prior_pos_enc = _PosEnc(D, D)
        self.prior_temporal_net = nn.TransformerDecoder(nn.TransformerDecoderLayer(D, 8, 512, 0.1), 1)
        self.mu_token = nn.Parameter(torch.zeros(D))
        self.logvar_token = nn.Parameter(torch.zeros(D))
        self.p_z_mu_net = nn.Linear(D, NZ)
        self.p_z_logvar_net = nn.Linear(D, NZ)


class MotionInfiller(nn.Module):
    def __init__(self):
        super().__init__()
        self.context_encoder = _InfillerContext()
        self.data_decoder = _InfillerDecoder()
        self.eval()

    def window(self, in_pose, key_pad, eps):
        """one 50-frame window: in_pose [50,B,69], key_pad [B,50] bool (True = ignore), eps [1|B,128] or None
        -> [40,B,69] (motion_infiller_vae.py:92-123, :345-398)"""
        ce, dd = self.context_encoder, self.data_decoder
        B = in_pose.shape[1]
        ctx = ce.temporal_net(ce.pos_enc(ce.in_fc(in_pose)), src_key_padding_mask=key_pad)
        tok = torch.cat([dd.mu_token.repeat(1, B, 1), dd.logvar_token.repeat(1, B, 1)], dim=0)
        px = dd.prior_temporal_net(dd.prior_pos_enc(tok), ctx, memory_key_padding_mask=key_pad)
        mu, logvar = dd.p_z_mu_net(px[0]), dd.p_z_logvar_net(px[1])
        z = mu + (eps if eps is not None else torch.randn_like(mu)) * torch.exp(0.5 * logvar)
        x = dd.temporal_net(dd.pos_enc(z.repeat(CUR, 1, 1), pos_offset=PAST), ctx, memory_key_padding_mask=key_pad)
        x = dd.out_fc(dd.out_mlp(x))
        return torch.cat([in_pose[:PAST], x], dim=0)

    @torch.no_grad()
    def inference(self, batch):
        """multi-step, sample_num 1 (:618-652): in_body_pose [B,T,69], frame_mask [B,T] (1 = visible),
        optional in_motion_latent [n_windows,128] -> infer_out_body_pose [B,1,T,69]"""
        dt = self.data_decoder.out_fc.weight.dtype                                       # float32 (reference); float64 in the fixture check
        pose = batch['in_body_pose'].transpose(0, 1).contiguous().to(dt).clone()         # [T,B,69]
        key_pad_all = ~(batch['frame_mask'] == 1)                                        # True where NOT visible
        T, B = pose.shape[0], pose.shape[1]
        W = PAST + CUR + FUT
        outs = []
        for i in range(int(np.ceil((T - PAST) / CUR))):
            s, e = i * CUR, i * CUR + W
            eb = min(e, T)
            win = pose[s:eb]
            kp = key_pad_all[:, s:eb]
            if e > eb:
                win = torch.cat([win, torch.zeros(e - eb, B, 69, dtype=dt)], dim=0)
                kp = torch.cat([kp, torch.ones(B, e - eb, dtype=torch.bool)], dim=1)
            kp = kp.clone()
            kp[:, :PAST] = False
            eps = batch['in_motion_latent'][[i]].to(dt) if 'in_motion_latent' in batch else None
            out = self.window(win, kp, eps)
            nfr = min(e - FUT, T) - s
            pose[s:s + nfr] = out[:nfr]
            outs.append(out[:nfr] if i == 0 else out[PAST:nfr])
        body = torch.cat(outs, dim=0).transpose(0, 1).unsqueeze(1).contiguous()          # [B,1,T,69]
        return {'infer_out_body_pose': body,
                'infer_out_pose': torch.cat([torch.zeros_like(body[..., :3]), body], dim=-1)}


class _TrajContext(nn.Module):
    def __init__(self):
        super().__init__()
        self.in_mlp = _MLP(69, [512, 256])
        self.temporal_net = nn.ModuleList([_BiLSTM(256, 256), _BiLSTM(256, 256)])
        self.out_mlp = _MLP(256, [512, 256])


class _TrajDecoder(nn.Module):
    def __init__(self):
        super().__init__()
        self.out_mlp = _MLP(256 + NZ, [512, 256])
        self.out_fc = nn.Linear(256, 11)
        self.prior_mlp = _MLP(256, [512, 256])
        self.p_z_net = nn.Linear(256, 2 * NZ)


class TrajPredictor(nn.Module):
    def __init__(self):
        super().__init__()
        self.context_encoder = _TrajContext()
        self.data_decoder = _TrajDecoder()
        self.eval()

    @torch.no_grad()
    def inference(self, joint_pos, eps=None, init_xy=None, init_heading=None):
        """joint_pos [T,B,69] -> local traj [T,B,11], trans [T,B,3], orient axis-angle [T,B,3]
        (traj_pred_vae.py:72-92, :281-333, :459-466)"""
        ce, dd = self.context_encoder, self.data_decoder
        x = ce.in_mlp(joint_pos)
        for net in ce.temporal_net:
            x = net(x)
        ctx = ce.out_mlp(x)
        mu, logvar = torch.chunk(dd.p_z_net(dd.prior_mlp(ctx.mean(dim=0))), 2, dim=-1)
        z = mu + (eps if eps is not None else torch.randn_like(mu)) * torch.exp(0.5 * logvar)
        out = dd.out_fc(dd.out_mlp(torch.cat([z.repeat(ctx.shape[0], 1, 1), ctx], dim=-1)))
        local = out.clone()
        local[0, :, :2] = 0.0 if init_xy is None else init_xy
        local[0, :, -2:] = torch.tensor([0.0, 1.0]) if init_heading is None else rt.heading_to_vec(init_heading)
        trans, q = tc.local_to_global(local)
        return local, trans, rt.quat_to_aa(q)


class MotionTrajJoint:
    """motion_traj_joint_model.py:141-145 with multi_step_mfiller=True, multi_step_trajpred=False, sample_num 1"""

    def __init__(self, state_mfiller, state_traj, smpl):
        self.mfiller, self.traj_predictor, self.smpl = MotionInfiller(), TrajPredictor(), smpl
        load_state(self.mfiller, state_mfiller)
        load_state(self.traj_predictor, state_traj)

    @torch.no_grad()
    def inference(self, batch, sample_num=1):
        assert sample_num == 1
        data = dict(batch)
        data.update(self.mfiller.inference(batch))
        body = data['infer_out_body_pose'][:, 0]                                          # [B,T,69]
        B, T = body.shape[:2]
        flat = body.reshape(-1, 69)
        z3 = torch.zeros_like(flat[:, :3])
        joints = self.smpl.get_joints(z3, flat, root_trans=z3)[:, 1:].reshape(B, T, 69).transpose(0, 1).contiguous()
        eps = batch['in_traj_latent'].to(body.dtype) if 'in_traj_latent' in batch else None
        local, trans, orient = self.traj_predictor.inference(joints, eps)
        data['infer_out_local_traj_tp'] = local.view(T, B, 1, 11)
        data['infer_out_trans'] = trans.transpose(0, 1).unsqueeze(1).contiguous()
        data['infer_out_orient'] = orient.transpose(0, 1).unsqueeze(1).contiguous()
        data['infer_out_pose'] = torch.cat([data['infer_out_orient'], data['infer_out_body_pose']], dim=-1)
        return data


def load_state(module, state):
    own = module.state_dict()
    missing = [k for k in own if k not in state]
    if missing:
        raise KeyError(f'missing parameters: {missing[:5]} ...')
    module.load_state_dict({k: torch.as_tensor(np.asarray(state[k])).float() for k in own}, strict=True)
