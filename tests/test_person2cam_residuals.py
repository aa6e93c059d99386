"""Per-person camera-relative residuals of the camera-from-persons mode (flag_opt_person2cam_rot / flag_opt_person2cam_trans,
global_recon_model.py:46-47,173-175,484-488,616-619): every frame's person2cam becomes person2cam @ [R(person2cam_res_rot) |
person2cam_res_trans] before the camera is averaged over the visible persons.

The analytic backward is checked against the oracle's autograd on the host-compiled frame functions and on the GPU, the
gradient of two gloo ranks against one rank, and the invariants: flag-off layout and launch count, zero gradient outside the
camera-from-persons mode, the struct size of the C ABI, and the refused regulariser."""
import copy
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import host_harness as hh
from emu_runner import EmuRunner
from glamr_b200 import lib as L
from glamr_b200 import problem as PB
from helpers import ReplayMT, case_setup
from oracle import rotations as rt
from oracle.global_opt import OracleGlobalRecon

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = ['3dpw_p2_t80_gaps', '3dpw_p1_t600_gaps']
P2C = ['person2cam_res_rot', 'person2cam_res_trans']
# On the 600-frame track the gradients of the scan roots traj_local_xy / traj_local_heading are sums of 600 per-frame terms that
# cancel down to the float32 rounding of those terms: two implementations (or the oracle in float32 and float64) agree there on
# no digit, and Adam turns that noise into lr-sized steps that the whole trajectory and the camera follow.  The track is
# compared on every other gradient at iteration 0 of each stage (the new blocks included); the step-by-step comparison runs on
# the 80-frame track, and the GPU test bounds the end state through the float64 continuation stored with the golden case.
LONG_TRACK = '3dpw_p1_t600_gaps'
SCAN_ROOTS = ('traj_local_xy', 'traj_local_heading')
PERSON_VARS = ['traj_local_xy', 'traj_local_dxy', 'traj_local_heading', 'traj_local_dheading', 'traj_local_z', 'traj_local_rot',
               'smpl_orient_world_res', 'root_trans_world_res', 'world_dheading'] + P2C


def _enable(cfg, rot, trans, stages):
    cfg.grecon_model_specs['flag_opt_person2cam_rot'] = rot
    cfg.grecon_model_specs['flag_opt_person2cam_trans'] = trans
    for st in stages:
        specs = cfg.opt_stage_specs[st]
        specs['opt_variables'] = list(specs['opt_variables']) + (['person2cam_rot'] if rot else []) + (['person2cam_trans'] if trans else [])


VARIANTS = {
    'rot_main': lambda cfg: _enable(cfg, True, False, ['main_opt']),
    'trans_main': lambda cfg: _enable(cfg, False, True, ['main_opt']),
    'both_all': lambda cfg: _enable(cfg, True, True, list(cfg.opt_stage_specs)),
}


def _setup(name, variant, smpl_assets):
    gold, cfg, in_dict = case_setup(name, smpl_assets)
    VARIANTS[variant](cfg)
    return gold, cfg, in_dict


class P2CEmuRunner(EmuRunner):
    """EmuRunner whose variable layout and problem compiler also see the two person2cam flags"""

    def __init__(self, oracle_model, data):
        self.model, self.data = oracle_model, data
        self.flags = {k: getattr(oracle_model, k) for k in
                      ['flag_fixed_cam', 'flag_opt_cam', 'flag_opt_cam_from_person_pose', 'flag_cam_inv_trans_res_all',
                       'flag_opt_vis_local_rot', 'cam_fix_frames', 'flag_opt_person2cam_rot', 'flag_opt_person2cam_trans']}
        self.layout = PB.make_layout(data, self.flags)
        self.theta = torch.zeros(self.layout.n_params)
        PB.bind_variables(data, self.layout, self.theta)
        self.comp = PB.StageCompiler(data, self.layout, self.flags, 'cpu', rt.aa_to_rot6d, aa_to_quat=rt.aa_to_quat)
        self.lib = hh.lib()
        self.h = None
        self.reduce = torch.zeros(self.layout.n_params + L.NUM_TERMS)


def _param_order(layout, vec, n_persons, model, opt_variables):
    """(name, view) of a packed [n_params] vector for every tensor of get_parameter, in its order (global_recon_model.py:591-633)"""
    gv = layout.views(vec)
    if 'cam' not in opt_variables:
        names = ['cam_inv_rot_residual', 'cam_inv_trans_residual']
    elif model.flag_fixed_cam:
        names = ['cam_rot_6d_fix', 'cam_trans_fix']
    else:
        names = ['cam_rot_6d', 'cam_trans']
    order = [(k, gv[k]) for k in names]
    for p in range(n_persons):
        pv = layout.views(vec, p)
        names = []
        for key in opt_variables:
            if key == 'world_res':
                names += ['smpl_orient_world_res', 'root_trans_world_res']
            if 'local' in key:
                names.append(f'traj_{key}')
        if model.flag_opt_person2cam_rot and 'person2cam_rot' in opt_variables:
            names.append('person2cam_res_rot')
        if model.flag_opt_person2cam_trans and 'person2cam_trans' in opt_variables:
            names.append('person2cam_res_trans')
        if 'world_dheading' in opt_variables:
            names.append('world_dheading')
        order += [(k, pv[k]) for k in names]
    return order


def _p2c_slots(model, opt_variables):
    """positions (within one person's block of get_parameter) of the person2cam variables this stage optimises"""
    return [k for k, f, v in [(P2C[0], model.flag_opt_person2cam_rot, 'person2cam_rot'),
                              (P2C[1], model.flag_opt_person2cam_trans, 'person2cam_trans')] if f and v in opt_variables]


def _oracle_grads(model, data, specs, stage):
    params = model.get_parameter(data, specs['opt_variables'])
    for p in params:
        p.requires_grad_(True)
        p.grad = None
    model.forward(data, specs['opt_variables'], {'stage': stage})
    total, _, uw = model.compute_loss(data, specs['loss_cfg'])
    total.backward()
    grads = [None if p.grad is None else p.grad.detach().clone() for p in params]
    for p in params:
        p.requires_grad_(False)
        p.grad = None
    return params, grads, {k: float(v) for k, v in uw.items()}, float(total)


def _hand_state(data_src, data_o):
    """the oracle continues from the implementation's variables and camera (the next stage is differentiated at identical
    variables; two independent Adam runs drift apart on these ill-conditioned tracks)"""
    for ps, po in zip(data_src['person_data'].values(), data_o['person_data'].values()):
        for k in PERSON_VARS:
            if k in ps:
                po[k] = ps[k].detach().cpu().clone()
    for k in ['cam_inv_rot_residual', 'cam_inv_trans_residual', 'cam_pose']:
        data_o[k] = data_src[k].detach().cpu().clone()
    data_o['cam_pose_inv'] = rt.inverse_transform(data_o['cam_pose'])


def _oracle_grads64(ora64, data_o, specs, stage):
    """the same closure evaluated in float64 from the same float32 state (OracleGlobalRecon.to_float64)"""
    return _oracle_grads(ora64, ora64.to_float64(data_o), specs, stage)[1]


def _check_grads(stage, order, grads, grads64, bound, skip=()):
    """|implementation - float64| within `bound` of the gradient's scale plus 4 x the float32 oracle's own deviation from
    float64.  `skip`: names not compared"""
    assert len(order) == len(grads)
    for (name, g_), gr, g64 in zip(order, grads, grads64):
        if gr is None:
            assert g_.numel() == 0 or float(g_.abs().max()) == 0.0, f'{stage} {name}: gradient where the oracle has none'
            continue
        if name in skip:
            continue
        g64 = g64.reshape(gr.shape)
        scale = max(float(g64.abs().max()), 1e-9)
        noise = float((gr.double() - g64).abs().max())
        err = float((g_.reshape(gr.shape).double() - g64).abs().max())
        assert err < bound * scale + 4.0 * noise, \
            f'{stage} grad of {name} {tuple(gr.shape)}: |err| {err:.2e} (scale {scale:.2e}, float32 oracle {noise:.2e})'


# ------------------------------------------------------------------------------------------------ host emulator
@pytest.mark.parametrize('variant', list(VARIANTS))
@pytest.mark.parametrize('name', CASES)
def test_emulator_matches_oracle_autograd(name, variant, smpl_assets):
    """every stage: iteration-0 term values and every variable's gradient (the new blocks included) vs the oracle's autograd,
    then the stage's Adam steps in both, with the bounds of test_globalopt_host_emu.py"""
    gold, cfg, in_dict = _setup(name, variant, smpl_assets)
    ora = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    data_o = ora.init_data(copy.deepcopy(in_dict))
    ora2 = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    data_e = ora2.init_data(copy.deepcopy(in_dict))
    ora64 = OracleGlobalRecon(cfg, smpl_assets)
    run = P2CEmuRunner(ora2, data_e)
    lay, P, T = run.layout, run.comp.P, run.comp.T
    assert lay.person2cam_res
    run.set_stage([], {}, 'init')
    run.backward()
    for stage, specs in cfg.opt_stage_specs.items():
        _hand_state(data_e, data_o)
        grads64 = _oracle_grads64(ora64, data_o, specs, stage)
        params, grads, uw, total = _oracle_grads(ora, data_o, specs, stage)
        run.set_stage(specs['opt_variables'], specs['loss_cfg'], stage)
        g_all, terms = run.backward()
        for k, v in uw.items():
            got = float(terms[L.TERM_INDEX[k]])
            assert abs(got - v) <= 2e-4 * max(abs(v), 1e-3) + 1e-7, f'{stage} term {k}: {got} vs {v}'
        assert abs(float(terms[-1]) - total) <= 2e-4 * abs(total) + 1e-6
        _check_grads(stage, _param_order(lay, run.reduce[:lay.n_params], P, ora2, specs['opt_variables']), grads, grads64, 3e-4,
                     skip=SCAN_ROOTS if name == LONG_TRACK else ())
        optimised = _p2c_slots(ora2, specs['opt_variables'])
        grad_of = {id(p_): g_ for p_, g_ in zip(params, grads)}
        for d in data_o['person_data'].values():
            for k in optimised:        # the comparison above is not vacuous: the camera really pulls on the residuals
                assert float(grad_of[id(d[k])].abs().max()) > 0.0, f'{stage} {k}: zero oracle gradient'
        before = {k: [lay.views(run.theta, p)[k].clone() for p in range(P)] for k in P2C}
        n = specs['opt_niters']
        if name == LONG_TRACK:          # the emulator takes the stage's steps; the next stage is compared at its variables
            for it in range(n):
                run.backward()
                run.step(specs['opt_lr'])
            for p in range(P):
                for k in P2C:
                    if k not in optimised:
                        assert torch.equal(lay.views(run.theta, p)[k], before[k][p]), f'{stage}: {k} moved although not optimised'
            cam = run.buffer(L.R_CAM_POSE).view(T, 3, 4)
            data_e['cam_pose'] = torch.cat([cam, torch.tensor([0., 0., 0., 1.]).expand(T, 1, 4)], dim=1).clone()
            continue
        loss_o, loss_e = [], []
        ora.optimize_main(data_o, specs['opt_variables'], specs['opt_lr'], n, specs['loss_cfg'], {'stage': stage},
                          on_iter=lambda it, last, dt: loss_o.append(float(last['loss'])))
        for it in range(n):
            _, terms = run.backward()
            loss_e.append(float(terms[-1]))
            run.step(specs['opt_lr'])
        np.testing.assert_allclose(loss_e, loss_o, rtol=2e-3, err_msg=f'{stage} loss trajectory')
        for p, d in enumerate(data_o['person_data'].values()):
            pv = lay.views(run.theta, p)
            for key in ['traj_local_xy', 'traj_local_heading', 'traj_local_rot', 'traj_local_dxy', 'traj_local_z', 'world_dheading'] + P2C:
                if key in d and id(d[key]) in grad_of and grad_of[id(d[key])] is not None:
                    g0 = grad_of[id(d[key])].reshape(pv[key].shape).abs()
                    sel = g0 > 1e-3 * g0.max()
                    diff = (pv[key] - d[key].detach().reshape(pv[key].shape)).abs()
                    tol = 2e-2 * specs['opt_lr'] * n + 1e-6
                    assert float(diff[sel].max()) < tol, f'{stage} after {n} steps: {key} differs by {float(diff[sel].max()):.2e}'
            for k in P2C:
                if k not in optimised:     # composed at its current value, but not moved by this stage's Adam
                    assert torch.equal(pv[k], before[k][p]), f'{stage}: {k} moved although the stage does not optimise it'
        cam = run.buffer(L.R_CAM_POSE).view(T, 3, 4)
        np.testing.assert_allclose(cam.numpy(), data_o['cam_pose'][:, :3, :].numpy(), atol=2e-4, err_msg=f'{stage} cam_pose')
        data_e['cam_pose'] = torch.cat([cam, torch.tensor([0., 0., 0., 1.]).expand(T, 1, 4)], dim=1).clone()


def test_emulator_residuals_inert_outside_camera_from_persons(smpl_assets):
    """flags on and the variables listed in every stage of a config whose camera is per-frame variables (glamr_dynamic): the
    residual does not enter the forward, its gradient is exactly zero in every stage (init included) and Adam leaves it at its
    initial value; every other gradient still matches the oracle"""
    gold, cfg, in_dict = case_setup('dynamic_p1_t40', smpl_assets)
    VARIANTS['both_all'](cfg)
    ora = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    data_o = ora.init_data(copy.deepcopy(in_dict))
    ora2 = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    run = P2CEmuRunner(ora2, ora2.init_data(copy.deepcopy(in_dict)))
    ora64 = OracleGlobalRecon(cfg, smpl_assets)
    lay, P = run.layout, run.comp.P
    init = run.theta.clone()
    p2c_blocks = [(lay.persons[p]['p2c_rot'], lay.persons[p]['p2c_trans'] + 3 * lay.T) for p in range(P)]
    run.set_stage([], {}, 'init')
    g, _ = run.backward()
    for a, b in p2c_blocks:
        assert float(g[a:b].abs().max()) == 0.0
    for stage, specs in cfg.opt_stage_specs.items():
        _hand_state(run.data, data_o)
        grads64 = _oracle_grads64(ora64, data_o, specs, stage)
        _, grads, _, _ = _oracle_grads(ora, data_o, specs, stage)
        run.set_stage(specs['opt_variables'], specs['loss_cfg'], stage)
        assert run.pb.cam_mode != L.CAM_FROM_PERSONS
        g, _ = run.backward()
        _check_grads(stage, _param_order(lay, run.reduce[:lay.n_params], P, ora2, specs['opt_variables']), grads, grads64, 3e-4)
        for a, b in p2c_blocks:
            assert float(g[a:b].abs().max()) == 0.0, f'{stage}: person2cam residual gradient outside camera mode 3'
        for it in range(specs['opt_niters']):
            run.backward()
            run.step(specs['opt_lr'])
        for a, b in p2c_blocks:
            assert torch.equal(run.theta[a:b], init[a:b]), f'{stage}: person2cam residual moved outside camera mode 3'
        cam = run.buffer(L.R_CAM_POSE).view(lay.T, 3, 4)
        run.data['cam_pose'] = torch.cat([cam, torch.tensor([0., 0., 0., 1.]).expand(lay.T, 1, 4)], dim=1).clone()


# ------------------------------------------------------------------------------------------------ 2 ranks (gloo)
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, name, ret):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    torch.set_num_threads(1)
    from glamr_b200.synthetic import make_smpl_assets
    assets = make_smpl_assets(0)
    gold, cfg, in_dict = _setup(name, 'both_all', assets)
    runs = {}
    for mode in ['single', 'sharded']:
        ora = OracleGlobalRecon(copy.deepcopy(cfg), assets, mt_model=ReplayMT(gold))
        runs[mode] = P2CEmuRunner(ora, ora.init_data(copy.deepcopy(in_dict)))
    single, sharded = runs['single'], runs['sharded']
    N = single.comp.P * single.comp.T
    lay = single.layout
    blocks = [slice(o['p2c_rot'], o['p2c_trans'] + 3 * lay.T) for o in lay.persons]
    g_err, p2c_err, p2c_scale = 0.0, 0.0, float('inf')
    for stage, specs in cfg.opt_stage_specs.items():
        single.set_stage(specs['opt_variables'], specs['loss_cfg'], stage)
        sharded.set_stage(specs['opt_variables'], specs['loss_cfg'], stage, n_begin=N * rank // world, n_end=N * (rank + 1) // world,
                          owner=(rank == 0))
        for it in range(3):
            # both evaluate the same variables: the single-rank run steps, the sharded one follows it (two Adam runs would
            # drift apart on the elements whose gradient is rounding noise)
            sharded.theta.copy_(single.theta)
            single.backward()
            sharded.backward()
            dist.all_reduce(sharded.reduce)              # the one collective per iteration
            a, b = single.reduce, sharded.reduce
            g_err = max(g_err, float((a - b).abs().max() / a.abs().max()))
            for s in blocks:   # the new entries on their own scale: each must be counted exactly once over the two ranks
                p2c_err = max(p2c_err, float((a[s] - b[s]).abs().max() / a[s].abs().max()))
                p2c_scale = min(p2c_scale, float(a[s].abs().max()))
            single.step(specs['opt_lr'])
    ret[rank] = (g_err, p2c_err, p2c_scale)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('name', CASES)
def test_sharded_gradient_equals_single_rank(name):
    """frame-persons split over two ranks by n_begin / n_end / owner (with one person, the person straddles the ranks), one
    all-reduce of [gradient | term sums] per iteration: equal to the single-rank buffer at the same variables, both stages,
    3 iterations each.  A person2cam entry counted twice or missed would be off by its whole value."""
    world, port = 2, _free_port()
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, name, ret), nprocs=world, join=True)
    for rank in range(world):
        g_err, p2c_err, p2c_scale = ret[rank]
        assert p2c_scale > 0.0, 'person2cam residual gradient is zero: nothing was checked'
        assert g_err < 1e-5, f'rank {rank}: reduced buffer differs from single-rank by {g_err:.2e} (relative)'
        assert p2c_err < 1e-4, f'rank {rank}: person2cam residual gradient differs from single-rank by {p2c_err:.2e} (relative)'


# ------------------------------------------------------------------------------------------------ invariants (CPU)
def _flags(rot, trans):
    return {'flag_fixed_cam': False, 'flag_opt_cam': True, 'flag_opt_cam_from_person_pose': True, 'flag_cam_inv_trans_res_all': True,
            'flag_opt_vis_local_rot': False, 'cam_fix_frames': [[0, None]], 'flag_opt_person2cam_rot': rot, 'flag_opt_person2cam_trans': trans}


def test_layout_with_flags_off_is_unchanged_and_new_blocks_come_last():
    T, lens, n_empty = 80, [80, 57], 5
    data = {'seq_len': T, 'fr_num_persons': torch.tensor([0] * n_empty + [1] * (T - n_empty)),
            'person_data': {i: {'exist_len': Ln} for i, Ln in enumerate(lens)}}
    base = PB.VariableLayout(T, n_empty, T, lens)
    off = PB.make_layout(data, _flags(False, False))
    legacy = {k: v for k, v in _flags(False, False).items() if 'person2cam' not in k}    # a flags dict that predates them
    expect = 9 * T + 9 + 6 * n_empty + 3 * T + sum(3 + 3 * (Ln - 1) + 7 * Ln + 7 * T for Ln in lens)
    for lay in (off, PB.make_layout(data, legacy)):
        assert not lay.person2cam_res
        assert lay.n_params == base.n_params == expect
        assert lay.persons == base.persons
        assert 'person2cam_res_rot' not in lay.views(torch.zeros(lay.n_params), 0)
    for rot, trans in [(True, False), (False, True), (True, True)]:
        on = PB.make_layout(data, _flags(rot, trans))
        assert on.n_params == expect + 9 * T * len(lens)
        for k in ['cam_rot', 'cam_trans', 'cam_rot_fix', 'cam_trans_fix', 'cam_inv_rot_res', 'cam_inv_trans_res']:
            assert getattr(on, k) == getattr(base, k)
        for p, (o_on, o_off) in enumerate(zip(on.persons, base.persons)):
            assert {k: v for k, v in o_on.items() if not k.startswith('p2c')} == o_off
            assert o_on['p2c_rot'] >= base.n_params and o_on['p2c_trans'] == o_on['p2c_rot'] + 6 * T
            v = on.views(torch.arange(on.n_params, dtype=torch.float32), p)
            assert v['person2cam_res_rot'].shape == (T, 6) and v['person2cam_res_trans'].shape == (T, 3)
            assert int(v['person2cam_res_rot'][0, 0]) == o_on['p2c_rot'] and int(v['person2cam_res_trans'][0, 0]) == o_on['p2c_trans']


def test_person_struct_size_unchanged():
    """the block offset lives in the former padding slot: the C struct and its ctypes mirror keep their size"""
    lib = hh.lib()
    lib.glamr_host_sizeof_person.restype = ctypes.c_size_t
    assert lib.glamr_host_sizeof_person() == ctypes.sizeof(L.Person) == 176
    assert L.Person.off_person2cam_res.offset == 11 * 4 and L.Person.traj_local_pred.offset == 12 * 4


def test_compiler_sets_offset_and_active_entries(smpl_assets):
    gold, cfg, in_dict = _setup('3dpw_p2_t80_gaps', 'rot_main', smpl_assets)
    ora = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    run = P2CEmuRunner(ora, ora.init_data(copy.deepcopy(in_dict)))
    lay, T = run.layout, run.comp.T
    for stage, specs in cfg.opt_stage_specs.items():
        pb = run.comp.compile(run.theta, specs['opt_variables'] + ['person2cam_trans'], specs['loss_cfg'], stage)
        persons = (L.Person * run.comp.P).from_buffer_copy(ctypes.string_at(pb.persons, ctypes.sizeof(L.Person) * run.comp.P))
        active = np.ctypeslib.as_array(ctypes.cast(pb.active, ctypes.POINTER(ctypes.c_uint8)), shape=(lay.n_params,))
        for p, o in enumerate(lay.persons):
            assert persons[p].off_person2cam_res == o['p2c_rot']
            assert active[o['p2c_rot']:o['p2c_rot'] + 6 * T].all() == (stage == 'main_opt')
            assert not active[o['p2c_trans']:o['p2c_trans'] + 3 * T].any()      # listed, but its flag is off
    ora = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    data = ora.init_data(copy.deepcopy(in_dict))
    ora.flag_opt_person2cam_rot = False
    off = P2CEmuRunner(ora, data)
    pb = off.comp.compile(off.theta, cfg.opt_stage_specs['main_opt']['opt_variables'], {}, 'main_opt')
    persons = (L.Person * off.comp.P).from_buffer_copy(ctypes.string_at(pb.persons, ctypes.sizeof(L.Person) * off.comp.P))
    assert all(persons[p].off_person2cam_res == -1 for p in range(off.comp.P))


def test_bind_variables_creates_missing_residuals():
    """a data dict without the variables (continued from a run without the flags) starts from the reference's init values"""
    T = 6
    data = {'seq_len': T, 'fr_num_persons': torch.ones(T, dtype=torch.int64), 'person_data': {0: {'exist_len': T}},
            'cam_inv_rot_residual': torch.zeros(0, 6), 'cam_inv_trans_residual': torch.zeros(T, 3)}
    lay = PB.make_layout(data, _flags(False, True))
    theta = torch.full((lay.n_params,), 7.0)
    PB.bind_variables(data, lay, theta)
    d = data['person_data'][0]
    assert torch.equal(d['person2cam_res_rot'], torch.tensor([1., 0., 0., 0., 1., 0.]).repeat(T, 1))
    assert torch.equal(d['person2cam_res_trans'], torch.zeros(T, 3))
    assert d['person2cam_res_rot'].data_ptr() == theta[lay.persons[0]['p2c_rot']:].data_ptr()


def test_person2cam_res_trans_reg_is_refused(smpl_assets):
    """the reference's regulariser looks the variable up in the top-level data dict and raises KeyError (as the oracle does):
    there is no behaviour to match, so the compiler refuses it with its own message"""
    from oracle.residuals import RESIDUALS
    gold, cfg, in_dict = _setup('3dpw_p2_t80_gaps', 'both_all', smpl_assets)
    ora = OracleGlobalRecon(cfg, smpl_assets, mt_model=ReplayMT(gold))
    data = ora.init_data(copy.deepcopy(in_dict))
    with pytest.raises(KeyError):
        RESIDUALS['person2cam_res_trans_reg'](data, {'weight': 1.0})
    run = P2CEmuRunner(ora, data)
    specs = cfg.opt_stage_specs['main_opt']
    with pytest.raises(NotImplementedError, match='person2cam_res_trans_reg.*fails in the reference'):
        run.comp.compile(run.theta, specs['opt_variables'], dict(specs['loss_cfg'], person2cam_res_trans_reg={'weight': 1.0}), 'main_opt')


# ------------------------------------------------------------------------------------------------ GPU
DEV = 'cuda:0'
EPS32 = 2.0 ** -24


def _noise_tol(gold, key, floor):
    """the bound test_gpu_parity.py puts on this output for the flag-off run of the same case: 4 x the reference's own float32
    noise (|ref32 - ref64|, |ref_pert - ref32|) + 32 float32 roundings of its magnitude, never tighter than `floor`"""
    r32, r64, rp = gold[f'final/{key}'], gold[f'final64/{key}'], gold[f'final_pert/{key}']
    noise = max(float(np.abs(r32 - r64).max()), float(np.abs(rp - r32).max()))
    return max(4.0 * noise + 32 * EPS32 * max(float(np.abs(r64).max()), 1.0), floor)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', list(VARIANTS))
@pytest.mark.parametrize('name', CASES)
def test_gpu_matches_oracle(name, variant, smpl_assets):
    """GlobalReconOptimizer: every stage's first closure (term values, every variable's gradient) vs the oracle's autograd at
    the bounds of test_unshipped_residual_terms_match_oracle_autograd; then optimize() end to end vs the oracle's optimize()"""
    from glamr_b200.recon import GlobalReconOptimizer
    gold, cfg, in_dict = _setup(name, variant, smpl_assets)
    model = GlobalReconOptimizer(cfg, torch.device(DEV), None, smpl=smpl_assets, mt_model=ReplayMT(gold, DEV))
    data = model.init_data(copy.deepcopy(in_dict))
    assert model._layout.person2cam_res
    ora = OracleGlobalRecon(copy.deepcopy(cfg), smpl_assets, mt_model=ReplayMT(gold))
    data_o = ora.init_data(copy.deepcopy(in_dict))
    ora64 = OracleGlobalRecon(copy.deepcopy(cfg), smpl_assets)
    for stage, specs in cfg.opt_stage_specs.items():
        grads64 = _oracle_grads64(ora64, data_o, specs, stage)
        _, grads, uw, _ = _oracle_grads(ora, data_o, specs, stage)
        model._cur_vars, model._cur_stage = specs['opt_variables'], stage
        model._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
        model._backward()
        with torch.cuda.device(DEV):
            L.check(model._lib.glamr_opt_losses(model._opt, L.ptr(model._reduce), L.ptr(model._terms), L.stream_ptr()), 'glamr_opt_losses')
        terms = model._terms.cpu().numpy()
        for k, v in uw.items():
            got = float(terms[L.TERM_INDEX[k]])
            assert abs(got - v) <= 3e-4 * max(abs(v), 1e-3) + 1e-7, f'{stage} term {k}: {got} vs {v}'
        grad = model._reduce[:model._layout.n_params].cpu()
        _check_grads(stage, _param_order(model._layout, grad, len(data['person_data']), model, specs['opt_variables']), grads, grads64, 5e-4,
                     skip=SCAN_ROOTS if name == LONG_TRACK else ())
        model.optimize_main(data, specs['opt_variables'], specs['opt_lr'], specs['opt_niters'], specs['loss_cfg'], {'stage': stage})
        _hand_state(data, data_o)
    # end to end: init_data + both stages, CUDA vs oracle, at the bounds of the golden 3dpw cases
    model = GlobalReconOptimizer(cfg, torch.device(DEV), None, smpl=smpl_assets, mt_model=ReplayMT(gold, DEV))
    out = model.optimize(copy.deepcopy(in_dict))
    ref = OracleGlobalRecon(copy.deepcopy(cfg), smpl_assets, mt_model=ReplayMT(gold)).optimize(copy.deepcopy(in_dict))
    cam_tol = _noise_tol(gold, 'cam_pose', 1e-4)
    err = float(np.abs(out['cam_pose'] - ref['cam_pose']).max())
    assert err <= cam_tol, f'cam_pose: {err:.3e} > {cam_tol:.3e}'
    for pid, pd in out['person_data'].items():
        pr = ref['person_data'][pid]
        for k in ['smpl_orient_world', 'root_trans_world', 'traj_local_xy', 'traj_local_dxy', 'traj_local_z', 'traj_local_rot',
                  'traj_local_heading', 'world_dheading', 'kp_2d_pred']:
            if k in pr and f'final64/{pid}/{k}' in gold:
                floor = 2e-2 if k == 'kp_2d_pred' else (1e-4 if k in ('smpl_orient_world', 'root_trans_world') else 0.0)
                tol = _noise_tol(gold, f'{pid}/{k}', floor)
                err = float(np.abs(pd[k].reshape(pr[k].shape) - pr[k]).max())
                assert err <= tol, f'{pid}/{k}: {err:.3e} > {tol:.3e}'
        # the residual as the transform it applies (its 6d scale directions have no gradient and random-walk under Adam in
        # both implementations): like the camera it shifts
        Ro, Rr = rt.rot6d_to_rotmat(torch.tensor(pd[P2C[0]])), rt.rot6d_to_rotmat(torch.tensor(pr[P2C[0]]))
        err = max(float((Ro - Rr).abs().max()), float(np.abs(pd[P2C[1]] - pr[P2C[1]]).max()))
        assert err <= cam_tol, f'{pid} person2cam residual: {err:.3e} > {cam_tol:.3e}'


@pytest.mark.gpu
def test_gpu_launch_count_and_other_camera_modes(smpl_assets):
    """the residuals add no launch; outside camera mode 3 (glamr_dynamic: per-frame camera variables) their gradient is exactly
    zero and optimize() returns them at their initial values"""
    from glamr_b200.recon import GlobalReconOptimizer
    counts = {}
    for variant in [None, 'both_all']:
        gold, cfg, in_dict = case_setup('3dpw_p2_t80_gaps', smpl_assets)
        if variant:
            VARIANTS[variant](cfg)
        model = GlobalReconOptimizer(cfg, torch.device(DEV), None, smpl=smpl_assets, mt_model=ReplayMT(gold, DEV))
        data = model.init_data(copy.deepcopy(in_dict))
        counts[variant] = [model.launches_per_iteration()]
        for stage, specs in cfg.opt_stage_specs.items():
            model._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
            counts[variant].append(model.launches_per_iteration())
    assert counts[None] == counts['both_all'], counts
    gold, cfg, in_dict = case_setup('dynamic_p1_t40', smpl_assets)
    VARIANTS['both_all'](cfg)
    model = GlobalReconOptimizer(cfg, torch.device(DEV), None, smpl=smpl_assets, mt_model=ReplayMT(gold, DEV))
    data = model.init_data(copy.deepcopy(in_dict))
    lay = model._layout
    blocks = [slice(o['p2c_rot'], o['p2c_trans'] + 3 * lay.T) for o in lay.persons]
    init = model._theta.clone()
    for stage, specs in cfg.opt_stage_specs.items():
        model._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
        assert model._pb.cam_mode != L.CAM_FROM_PERSONS
        model._backward()
        for s in blocks:
            assert float(model._reduce[s].abs().max()) == 0.0, f'{stage}: person2cam residual gradient outside camera mode 3'
        model.optimize_main(data, specs['opt_variables'], specs['opt_lr'], specs['opt_niters'], specs['loss_cfg'], {'stage': stage})
        for s in blocks:
            assert torch.equal(model._theta[s], init[s]), f'{stage}: person2cam residual moved outside camera mode 3'
    d = data['person_data'][0]
    assert torch.equal(d['person2cam_res_rot'].cpu(), torch.tensor([1., 0., 0., 0., 1., 0.]).repeat(lay.T, 1))
