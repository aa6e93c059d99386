"""Live per-kernel timing of one optimiser iteration (CUDA events between launches, eager mode)."""
import copy, ctypes, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from glamr_b200 import lib as L
from glamr_b200.config import Config
from glamr_b200.recon import GlobalReconOptimizer
from glamr_b200.smpl import SMPL
from glamr_b200.synthetic import make_in_dict, make_smpl_assets, SyntheticPrior
P, T = int(os.environ.get('P', 1)), int(os.environ.get('T', 300))
cfgid = os.environ.get('CFG', 'glamr_dynamic')
a = make_smpl_assets(0); dev = torch.device('cuda:0')
cfg = Config(cfgid); in_dict = make_in_dict(a, P, T)
m = GlobalReconOptimizer(cfg, dev, None, smpl=SMPL(a, device=dev), mt_model=SyntheticPrior(0, dev))
data = m.init_data(copy.deepcopy(in_dict))
stage, specs = list(cfg.opt_stage_specs.items())[-1]
m._cur_vars, m._cur_stage, m._loss_cfg = specs['opt_variables'], stage, specs['loss_cfg']
m._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
hist = torch.zeros((400, L.NUM_TERMS + 1), device=dev)
lib = m._lib
def it():      # the library's single-GPU iteration (forward, LBS, residuals, backward, Adam), eager so that events can sit between launches
    L.check(lib.glamr_opt_iterate(m._opt, L.ptr(m._theta), L.ptr(m._reduce), float(specs['opt_lr']), L.ptr(hist), L.NUM_TERMS + 1, 1, 0, L.stream_ptr()), 'iterate')
for _ in range(5): it()
L.check(lib.glamr_opt_kernel_timing(m._opt, 2), 't')
acc = None
for _ in range(50):
    it()
    ms = (ctypes.c_float * 24)(); n = ctypes.c_int()
    L.check(lib.glamr_opt_kernel_times(m._opt, ms, ctypes.byref(n)), 'times')
    v = np.array(ms[:n.value]); acc = v if acc is None else acc + v
acc = acc / 50 * 1000
print(f'P={P} T={T} {cfgid}:{stage}  per-segment us:', np.round(acc, 1).tolist(), 'sum', round(float(acc.sum()), 1))
