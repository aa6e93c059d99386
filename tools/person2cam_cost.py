"""Per-iteration cost of the person2cam residuals (flag_opt_person2cam_rot / _trans) in the camera-from-persons mode.

For the golden glamr_3dpw tracks (2 persons x 80 frames, 1 person x 600 frames) the main_opt iteration (glamr_opt_iterate:
one replayed CUDA graph per iteration, L2 flushed before each, CUDA events around it) is timed with the flags off and on
(both residual blocks optimised), and with the flags off through a second library build (--other-so, e.g. the parent
commit's).  Every configuration runs in a process of its own; the configurations alternate run by run.  Prints the GPU,
its power limit, one JSON line per run and the median and range over runs of the per-run median.

    python tools/person2cam_cost.py [--runs 6] [--iters 300] [--other-so path/to/libglamr_b200.so] [--out DIR]
"""
import argparse
import copy
import hashlib
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ['3dpw_p2_t80_gaps', '3dpw_p1_t600_gaps']


def child(case, flags_on, iters):
    sys.path[:0] = [REPO, os.path.join(REPO, 'tests')]
    import numpy as np
    import torch
    from glamr_b200 import lib as L
    from glamr_b200.recon import GlobalReconOptimizer
    from glamr_b200.synthetic import make_smpl_assets
    from helpers import ReplayMT, case_setup
    assets = make_smpl_assets(0)
    gold, cfg, in_dict = case_setup(case, assets)
    stage, specs = 'main_opt', cfg.opt_stage_specs['main_opt']
    if flags_on:
        cfg.grecon_model_specs.update(flag_opt_person2cam_rot=True, flag_opt_person2cam_trans=True)
        specs['opt_variables'] = list(specs['opt_variables']) + ['person2cam_rot', 'person2cam_trans']
    dev = torch.device('cuda:0')
    m = GlobalReconOptimizer(cfg, dev, None, smpl=assets, mt_model=ReplayMT(gold, dev))
    data = m.init_data(copy.deepcopy(in_dict))
    m._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
    terms = torch.zeros(L.NUM_TERMS + 1, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def it():
        L.check(m._lib.glamr_opt_iterate(m._opt, L.ptr(m._theta), L.ptr(m._reduce), float(specs['opt_lr']), L.ptr(terms), 0, 1, 1,
                                         L.stream_ptr()), 'glamr_opt_iterate')
    for _ in range(30):
        it()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        flush.fill_(1)                 # evict L2 (126 MB) before every timed iteration
        a.record()
        it()
        b.record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in evs])
    # the variables after the same iteration count: with the flags off both builds must agree bit for bit
    theta = m._theta.cpu().numpy().tobytes()
    return {'case': case, 'flags_on': flags_on, 'so': os.environ.get('GLAMR_B200_SO', 'tree'), 'median_us': float(np.median(ms) * 1e3),
            'launches': m.launches_per_iteration(), 'n_params': m._layout.n_params, 'theta_sha256': hashlib.sha256(theta).hexdigest()[:16]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--runs', type=int, default=6)
    ap.add_argument('--iters', type=int, default=300)
    ap.add_argument('--other-so', default=None)
    ap.add_argument('--out', default=None)
    ap.add_argument('--child', default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        case, on = args.child.split(',')
        print(json.dumps(child(case, on == '1', args.iters)))
        return
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print('gpu:', gpu)
    configs = [('this build, flags off', None, 0), ('this build, flags on', None, 1)]
    if args.other_so:
        configs.insert(0, ('other build, flags off', os.path.abspath(args.other_so), 0))
    rows = []
    for r in range(args.runs):
        for case in CASES:
            for label, so, on in configs:
                env = dict(os.environ)
                env.pop('GLAMR_B200_SO', None)
                if so:
                    env['GLAMR_B200_SO'] = so
                out = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', f'{case},{on}', '--iters', str(args.iters)],
                                     env=env, capture_output=True, text=True, cwd=REPO)
                if out.returncode != 0:
                    sys.exit(out.stdout + out.stderr)
                res = dict(json.loads(out.stdout.strip().splitlines()[-1]), run=r, label=label)
                print(json.dumps(res), flush=True)
                rows.append(res)
    summary = {'gpu': gpu}
    for case in CASES:
        off = {x['theta_sha256'] for x in rows if x['case'] == case and not x['flags_on']}
        summary[f'{case} | flags-off variables identical across builds and runs'] = len(off) == 1
    for case in CASES:
        for label, _, _ in configs:
            v = sorted(x['median_us'] for x in rows if x['case'] == case and x['label'] == label)
            summary[f'{case} | {label}'] = {'median_us': v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2]),
                                            'min_us': v[0], 'max_us': v[-1], 'runs': len(v)}
    print(json.dumps(summary, indent=1))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'person2cam_cost.json'), 'w') as f:
            json.dump({'runs': rows, 'summary': summary}, f, indent=1)


if __name__ == '__main__':
    main()
