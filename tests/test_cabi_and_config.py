"""CPU-only checks: the C-ABI library exports every symbol include/glamr_b200.h declares (no compute calls), struct
layouts agree with the ctypes mirror, the built-in stage tables equal the reference YAML, the product refuses CPU."""
import ctypes
import json
import numpy as np
import os

import pytest
import torch

import __graft_entry__ as ge
from conftest import GOLDEN
from glamr_b200 import lib as L
from glamr_b200.config import BUILTIN_IDS, Config, builtin_config_dict


@pytest.fixture(scope='module')
def cdll():
    ge.build()
    return ctypes.CDLL(L.SO_PATH)


def test_library_exports_every_declared_symbol(cdll):
    syms = ge.exported_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(cdll, s), s


def test_struct_layouts_match(cdll):
    cdll.glamr_sizeof_person.restype = ctypes.c_size_t
    cdll.glamr_sizeof_problem.restype = ctypes.c_size_t
    assert cdll.glamr_sizeof_person() == ctypes.sizeof(L.Person)
    assert cdll.glamr_sizeof_problem() == ctypes.sizeof(L.Problem)
    assert cdll.glamr_version() >= 100


def test_term_table_matches_header():
    hdr = open(os.path.join(os.path.dirname(L.HERE), 'include', 'glamr_b200.h')).read()
    body = hdr[hdr.index('enum glamr_term {'):hdr.index('GLAMR_NUM_TERMS')]
    names = [n.strip().split('=')[0].strip() for n in body.split('{')[1].split(',') if n.strip()]
    assert len(names) == L.NUM_TERMS == len(L.TERM_INDEX)


def test_product_requires_cuda_device():
    with pytest.raises(L.GlamrError):
        L.require_cuda('cpu')


@pytest.mark.parametrize('cfg_id', BUILTIN_IDS)
def test_builtin_configs_equal_reference_yaml(cfg_id):
    """tests/golden/configs.json: the reference's global_recon/cfg/<cfg_id>.yml as parsed by yaml.safe_load"""
    with open(os.path.join(GOLDEN, 'configs.json')) as f:
        ref = json.load(f)[cfg_id]
    mine = builtin_config_dict(cfg_id)
    assert mine['grecon_model_specs'] == ref['grecon_model_specs']
    assert mine['opt_stage_specs'] == ref['opt_stage_specs']
    assert mine['grecon_model_name'] == ref['grecon_model_name'] and mine['dataset'] == ref['dataset']


def test_config_surface():
    cfg = Config('glamr_static_multi', out_dir='/tmp/glamr_b200_cfg_test')
    assert cfg.id == 'glamr_static_multi' and cfg.grecon_model_name == 'global_recon_model'
    assert list(cfg.opt_stage_specs) == ['init_opt', 'main_opt'] and cfg.grecon_model_specs['flag_fixed_cam'] is True


def test_rotmats_to_rotvec_matches_scipy():
    """host step of init_data (global_recon_model.py:106-107): float32 rotation matrices -> rotation vectors"""
    from scipy.spatial.transform import Rotation
    from glamr_b200.recon import rotmats_to_rotvec
    rng = np.random.default_rng(0)
    rv = rng.normal(size=(4000, 3)) * rng.uniform(0, 1.5, size=(4000, 1))
    rv[:50] *= 1e-5                                                                       # series branch
    rv[50:100] = rv[50:100] / np.linalg.norm(rv[50:100], axis=1, keepdims=True) * (np.pi - 1e-4)   # near pi
    mats = Rotation.from_rotvec(rv).as_matrix().astype(np.float32)                        # float32-accurate, as HybrIK stores them
    np.testing.assert_allclose(rotmats_to_rotvec(mats), Rotation.from_matrix(mats).as_rotvec(), atol=1e-10)


def test_tensor_to_numpy_batched_copy_keeps_values_shapes_dtypes(monkeypatch):
    """output conversion of optimize() (lib/utils/torch_utils.py:118): grouped device->host copies, same nested structure"""
    from glamr_b200 import recon
    g = torch.Generator().manual_seed(0)
    data = {'a': torch.randn(3, 4, generator=g), 'flag': True, 'name': 'seq', 'n': 7, 'none': None,
            'person_data': {0: {'x': torch.randn(5, generator=g), 'mask': torch.tensor([True, False, True]), 'k': torch.arange(6).reshape(2, 3),
                                'd': torch.randn(2, 2, generator=g).double(), 'empty': torch.zeros(0, 6), 'scalar': torch.tensor(2.5)}},
            'rel': {(0, 1): torch.randn(2, 4, 4, generator=g)}, 'lst': [torch.ones(2), (torch.zeros(1), 3)]}
    # force the grouped path for CPU tensors too (on the product path the tensors are CUDA tensors)
    monkeypatch.setattr(recon, '_GROUP_CPU_TENSORS', True, raising=False)
    out = recon.tensor_to_numpy(data)

    def check(a, b):
        if isinstance(a, torch.Tensor):
            assert isinstance(b, np.ndarray) and b.shape == tuple(a.shape) and b.dtype == a.numpy().dtype
            np.testing.assert_array_equal(b, a.numpy())
        elif isinstance(a, dict):
            assert list(a.keys()) == list(b.keys())
            for k in a:
                check(a[k], b[k])
        elif isinstance(a, (list, tuple)):
            assert type(a) is type(b) and len(a) == len(b)
            for u, v in zip(a, b):
                check(u, v)
        else:
            assert a is b or a == b
    check(data, out)


def test_load_smpl_assets_official_pickle_layout(tmp_path):
    """on-disk SMPL model as smplx reads it (lib/models/smpl.py:274-279 -> smplx.SMPL.__init__): sparse J_regressor,
    posedirs [6890,3,207], 300 shape components, kintree_table with 2^32-1 as the root's parent, faces under 'f'"""
    import pickle
    import scipy.sparse as sp
    from glamr_b200.smpl import load_smpl_assets
    rng = np.random.default_rng(0)
    V = 6890
    jr = np.zeros((24, V), np.float64)
    for j in range(24):
        idx = rng.choice(V, 8, replace=False)
        jr[j, idx] = rng.dirichlet(np.ones(8))
    parents = np.array([4294967295, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21], dtype=np.uint32)
    model = {'v_template': rng.normal(size=(V, 3)), 'shapedirs': rng.normal(size=(V, 3, 300)).astype(np.float32),
             'posedirs': rng.normal(size=(V, 3, 207)).astype(np.float32), 'J_regressor': sp.csc_matrix(jr),
             'weights': rng.random((V, 24)), 'kintree_table': np.stack([parents, np.arange(24, dtype=np.uint32)]),
             'f': rng.integers(0, V, size=(13776, 3)).astype(np.uint32)}
    d = tmp_path / 'smpl'
    d.mkdir()
    with open(d / 'SMPL_NEUTRAL.pkl', 'wb') as fh:
        pickle.dump(model, fh)
    np.save(tmp_path / 'J_regressor_extra.npy', rng.random((9, V)))
    a = load_smpl_assets(str(d), str(tmp_path / 'J_regressor_extra.npy'))
    assert a['shapedirs'].shape == (V, 3, 10) and a['posedirs'].shape == (207, V * 3) and a['J_regressor'].shape == (24, V)
    assert a['lbs_weights'].shape == (V, 24) and a['faces'].shape == (13776, 3) and a['J_regressor_extra'].shape == (9, V)
    assert list(a['parents'][:4]) == [-1, 0, 0, 0]
    # smplx: posedirs.reshape(-1, 207).T -> row k holds the offsets of every (vertex, coordinate) for pose feature k
    np.testing.assert_array_equal(a['posedirs'][5].reshape(V, 3), model['posedirs'][:, :, 5])
    np.testing.assert_allclose(a['J_regressor'], jr)


def test_checkpoint_discovery_follows_reference_layout(tmp_path):
    """lib/utils/tools.py:41-45,94-104: results/<cfg>/version_<latest>/checkpoints/*best*.ckpt"""
    from glamr_b200.motion_traj import _find_checkpoint
    root = tmp_path / 'results' / 'motion_filler' / 'motion_infiller_demo'
    for v, names in {0: ['model-best-epoch=0003.ckpt'], 2: ['last.ckpt'], 10: ['model-best-epoch=0040.ckpt', 'last.ckpt']}.items():
        d = root / f'version_{v}' / 'checkpoints'
        d.mkdir(parents=True)
        for n in names:
            (d / n).write_bytes(b'')
    assert _find_checkpoint(str(root)).endswith(os.path.join('version_10', 'checkpoints', 'model-best-epoch=0040.ckpt'))   # numeric, not lexical, order
    with pytest.raises(FileNotFoundError):
        _find_checkpoint(str(tmp_path / 'results' / 'traj_pred' / 'traj_pred_demo'))
