import os, sys, torch, time
sys.path.insert(0, '.')
from glamr_b200.smpl import SMPL
from glamr_b200.synthetic import make_smpl_assets
a = make_smpl_assets(0)
smpl = SMPL(a, device='cuda:0')
n = int(os.environ.get('N', 300))
g = torch.Generator().manual_seed(0)
o, p, b, t = [x.cuda() for x in (torch.randn(n,3,generator=g), torch.randn(n,69,generator=g)*0.3, torch.randn(n,10,generator=g), torch.randn(n,3,generator=g))]
for _ in range(5): smpl(global_orient=o, body_pose=p, betas=b, root_trans=t, return_verts=False)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
K = 50
e0.record()
for _ in range(K): smpl(global_orient=o, body_pose=p, betas=b, root_trans=t, return_verts=False)
e1.record(); torch.cuda.synchronize()
print('N', n, 'dbg', os.environ.get('GLAMR_LBS_DEBUG'), 'us per smpl forward', e0.elapsed_time(e1)/K*1000)
