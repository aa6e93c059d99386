"""Small end-to-end case for compute-sanitizer (memcheck / racecheck): SMPL forward at a ragged size through both LBS paths,
one prior inference, and a short optimisation through the iteration kernels.

    compute-sanitizer --tool memcheck  python tools/sanitize_case.py
    compute-sanitizer --tool racecheck python tools/sanitize_case.py
"""
import copy
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from glamr_b200 import lib as L
from glamr_b200.config import Config
from glamr_b200.motion_traj import MotionTrajJointModel
from glamr_b200.recon import GlobalReconOptimizer
from glamr_b200.smpl import SMPL
from glamr_b200.synthetic import LatentInjector, make_in_dict, make_smpl_assets
from glamr_b200.synthetic_nets import make_prior_states

dev = torch.device('cuda:0')
a = make_smpl_assets(0)
smpl = SMPL(a, device=dev)
g = torch.Generator().manual_seed(0)
n = 33
for path in (2, 1, 0):
    L.check(L.load().glamr_smpl_set_lbs_path(path), 'path')
    out = smpl(global_orient=torch.randn(n, 3, generator=g).to(dev), body_pose=(torch.randn(n, 69, generator=g) * 0.3).to(dev),
               betas=torch.randn(n, 10, generator=g).to(dev), root_trans=torch.randn(n, 3, generator=g).to(dev))
    torch.cuda.synchronize()
    print('smpl path', path, float(out.vertices.abs().sum()))
L.check(L.load().glamr_smpl_set_lbs_path(-1), 'path')        # back to the default for the optimiser runs below
prior = MotionTrajJointModel(None, dev, None, smpl=smpl, states=make_prior_states(1234))
which = os.environ.get('CASES', 'glamr_dynamic,glamr_static_multi,glamr_3dpw').split(',')
for cfg_id in which:
    P = 2 if 'multi' in cfg_id or '3dpw' in cfg_id else 1
    cfg = Config(cfg_id)
    for st in cfg.opt_stage_specs.values():
        st['opt_niters'] = 3
    in_dict = make_in_dict(a, P, 40, seed=1, gaps='3dpw' in cfg_id)
    m = GlobalReconOptimizer(cfg, dev, None, smpl=smpl, mt_model=LatentInjector(prior, 0))
    out = m.optimize(copy.deepcopy(in_dict))
    torch.cuda.synchronize()
    print(cfg_id, 'ok', float(out['cam_pose'].sum()))
print('sanitize case done')
