"""ctypes binding of the CUDA library (include/glamr_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a) as ``glamr_b200/libglamr_b200.so``.
There is no CPU fallback: ``load()`` raises if the shared object is missing, and every call raises on a non-zero
return code.
"""
import ctypes
import os
import subprocess

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
# GLAMR_B200_SO: tools/ only -- load another build of the same sources (the -DGLAMR_EXPERIMENT library with the work-skipping switches and
# section stamps); bench.py refuses to run with it set
REL_SO_PATH = os.path.join(HERE, 'libglamr_b200.so')
SO_PATH = os.environ.get('GLAMR_B200_SO') or REL_SO_PATH
EXP_SO_PATH = os.path.join(HERE, 'libglamr_b200_exp.so')
CSRC = os.path.join(HERE, 'csrc')
SOURCES = ['smpl_kernels.cu', 'globalopt_kernels.cu', 'c_api.cu', 'nets_kernels.cu', 'eval_kernels.cu']
NUM_TERMS = 21

TERM_INDEX = {
    'kp_2d': 0, 'kp_2d_dist': 1, 'cam_traj_rot': 2, 'cam_traj_trans': 3, 'traj_rot_smoothness': 4,
    'traj_trans_smoothness': 5, 'rel_transform': 6, 'local_traj_dxy_reg': 7, 'local_traj_dheading_reg': 8,
    'local_traj_dheading_reg_new': 9, 'local_traj_rot_reg': 10, 'local_traj_z_reg': 11, 'traj_rot_res': 12,
    'traj_trans_res': 13, 'cam_inv_trans_residual_reg': 14, 'cam_inv_rot_smoothness': 15, 'cam_origin_smoothness': 16,
    'cam_up_reg': 17, 'cam_rot_smoothness': 18, 'cam_trans_smoothness': 19, 'cam_depth_smoothness': 20,
}
CAM_CONST, CAM_PER_FRAME, CAM_FIXED, CAM_FROM_PERSONS = 0, 1, 2, 3
(R_ORIENT_WORLD, R_TRANS_WORLD, R_ORIENT_BASE, R_TRANS_BASE, R_KP_PRED, R_ORIENT_CIW, R_TRANS_CIW, R_CAM_POSE,
 R_CAM_POSE_INV, R_JOINTS_WORLD, R_TRAJ_LOCAL) = range(11)

# rowops.cuh
(ROP_AA_TO_ROTMAT, ROP_RODRIGUES_SMPLX, ROP_ROT6D_TO_ROTMAT, ROP_ROTMAT_TO_QUAT, ROP_QUAT_TO_AA, ROP_AA_TO_QUAT,
 ROP_QUAT_MUL, ROP_ROTMAT_TO_AA, ROP_QUAT_TO_ROTMAT, ROP_SAFE_ATAN2, ROP_PROJECT, ROP_MAT3_MUL) = range(12)
ROP_DIMS = {0: (3, 0, 9), 1: (3, 0, 9), 2: (6, 0, 9), 3: (9, 0, 4), 4: (4, 0, 3), 5: (3, 0, 4), 6: (4, 4, 4), 7: (9, 0, 3),
            8: (4, 0, 9), 9: (2, 0, 1), 10: (3, 9, 2), 11: (9, 9, 9)}

_fp = ctypes.POINTER(ctypes.c_float)
_vp = ctypes.c_void_p


class Person(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ['start', 'len', 'off_xy', 'off_heading', 'off_dxy', 'off_dheading', 'off_z', 'off_rot',
                 'off_world_dheading', 'off_orient_res', 'off_trans_res', 'off_person2cam_res']] + \
               [(n, _vp) for n in
                ['traj_local_pred', 'orient_base_init', 'trans_base_init', 'cam_K', 'kp_target', 'orient_cam_6d',
                 'orient_cam_q', 'trans_cam', 'person2cam', 'dheading_mask', 'rot_mask', 'vis', 'kp_w', 'kp_dist_mask', 'ctr_w', 'ctt_w']]


class Problem(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ['P', 'T', 'J', 'cam_mode', 'off_cam_rot', 'off_cam_trans', 'use_world_res', 'has_world_dheading',
                 'trans_res_all', 'cam_up_first_only', 'n_params', 'n_begin', 'n_end', 'owner', 'cam_traj_rot_quat', 'traj_rot_smooth_quat']] + \
               [('cam_up_first_weight', ctypes.c_float), ('rel_trans_weight', ctypes.c_float),
                ('term_weight', ctypes.c_float * NUM_TERMS), ('term_norm', ctypes.c_float * NUM_TERMS),
                ('term_enabled', ctypes.c_int32 * NUM_TERMS), ('term_monitor', ctypes.c_int32 * NUM_TERMS)] + \
               [(n, _vp) for n in
                ['persons', 'smpl_pose_all', 'smpl_beta_all', 'scale_all', 'cam_pose_const', 'empty_index', 'fill_src',
                 'inv_num_persons', 'rel_target', 'rel_w', 'rel_wt', 'active']]


class GlamrError(RuntimeError):
    pass


_lib = None


def nvcc_command(out_path=None, experiment=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    return ['nvcc', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
            '-Xcompiler', '-fPIC', '-shared'] + (['-DGLAMR_EXPERIMENT'] if experiment else []) + \
           ['-o', out_path or (EXP_SO_PATH if experiment else REL_SO_PATH)] + srcs


def build_experiment():
    """the -DGLAMR_EXPERIMENT variant for tools/ (never loaded by default)"""
    res = subprocess.run(nvcc_command(experiment=True), capture_output=True, text=True)
    if res.returncode != 0:
        raise GlamrError('nvcc failed:\n' + res.stdout + res.stderr)
    return EXP_SO_PATH


def build(force=False, verbose=False):
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'glamr_b200.h')]
    newest = max(os.path.getmtime(p) for p in srcs)
    if not force and os.path.exists(REL_SO_PATH) and os.path.getmtime(REL_SO_PATH) >= newest:
        return REL_SO_PATH
    cmd = nvcc_command()
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise GlamrError('nvcc failed:\n' + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return REL_SO_PATH


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise GlamrError(f'{SO_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"`. '
                         'glamr_b200 has no CPU fallback.')
    lib = ctypes.CDLL(SO_PATH)
    lib.glamr_smpl_workspace_bytes.restype = ctypes.c_size_t
    lib.glamr_smpl_fk_workspace_bytes.restype = ctypes.c_size_t
    lib.glamr_sizeof_person.restype = ctypes.c_size_t
    lib.glamr_sizeof_problem.restype = ctypes.c_size_t
    lib.glamr_opt_reduce_count.restype = ctypes.c_size_t
    lib.glamr_opt_peer_bytes.restype = ctypes.c_size_t
    lib.glamr_fp32_probe.argtypes = [ctypes.c_int, _vp, ctypes.c_size_t, _vp, _vp]
    lib.glamr_opt_last_lbs_parts_ms.argtypes = [_vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    lib.glamr_opt_time_blend.argtypes = [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    lib.glamr_peer_alloc.argtypes = [ctypes.c_size_t, _vp, _vp]
    lib.glamr_peer_open.argtypes = [_vp, _vp]
    lib.glamr_peer_close.argtypes = [_vp]
    lib.glamr_peer_free.argtypes = [_vp]
    lib.glamr_opt_set_peers.argtypes = [_vp, ctypes.c_int, ctypes.c_int, _vp]
    lib.glamr_allreduce_inplace.argtypes = [_vp, _vp, ctypes.c_size_t, _vp]
    lib.glamr_opt_apply.argtypes = [_vp, _vp, _vp, ctypes.c_double, _vp, ctypes.c_int, _vp]
    lib.glamr_opt_iterate.argtypes = [_vp, _vp, _vp, ctypes.c_double, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]
    if lib.glamr_sizeof_person() != ctypes.sizeof(Person) or lib.glamr_sizeof_problem() != ctypes.sizeof(Problem):
        raise GlamrError('struct layout mismatch between include/glamr_b200.h and glamr_b200/lib.py')
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        if rc > 0:
            raise GlamrError(f'{what}: CUDA error {rc}')
        raise GlamrError(f'{what}: {({-1: "invalid argument", -2: "workspace too small", -3: "unsupported"}).get(rc, rc)}')


def ptr(t):
    """device pointer of a contiguous tensor (or None)"""
    if t is None:
        return None
    assert t.is_contiguous(), 'tensor must be contiguous'
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(device):
    device = torch.device(device)
    if device.type != 'cuda':
        raise GlamrError('glamr_b200 runs on CUDA devices only (no CPU fallback); got device ' + str(device))
    if not torch.cuda.is_available():
        raise GlamrError('no CUDA device available')
    return device


def rowop(op, a, b=None):
    """out rows = op(a rows[, b rows]) on the CUDA library; a, b: float32 cuda tensors [..., d]"""
    d0, d1, do = ROP_DIMS[op]
    a2 = a.reshape(-1, d0).contiguous().float()
    b2 = None if b is None else b.reshape(-1, d1).contiguous().float()
    out = torch.empty((a2.shape[0], do), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        check(load().glamr_rowop_fwd(op, a2.shape[0], ptr(a2), ptr(b2), ptr(out), stream_ptr()), 'glamr_rowop_fwd')
    return out.reshape(a.shape[:-1] + (do,))


def rowop_vjp(op, a, b, g, want_b=False):
    d0, d1, do = ROP_DIMS[op]
    a2 = a.reshape(-1, d0).contiguous().float()
    b2 = None if b is None else b.reshape(-1, d1).contiguous().float()
    g2 = g.reshape(-1, do).contiguous().float()
    ga = torch.empty_like(a2)
    gb = torch.empty_like(b2) if (want_b and b2 is not None) else None
    with torch.cuda.device(a.device):
        check(load().glamr_rowop_vjp(op, a2.shape[0], ptr(a2), ptr(b2), ptr(g2), ptr(ga), ptr(gb), stream_ptr()), 'glamr_rowop_vjp')
    return ga.reshape(a.shape), (None if gb is None else gb.reshape(b.shape))
