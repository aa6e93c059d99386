"""bench.py --dump-outputs: what the last timed step computed, written as DIR/<name>.npy so that two builds run with the same
arguments can be compared output for output."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def bench():
    argv = sys.argv
    sys.argv = ['bench.py']
    try:
        spec = importlib.util.spec_from_file_location('bench_dump_under_test', os.path.join(REPO, 'bench.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


class _Model:
    """stands in for GlobalReconOptimizer: packed variables plus the per-frame outputs _scatter_outputs refreshes"""

    def __init__(self, bench, P, T):
        g = torch.Generator().manual_seed(0)
        self._theta = torch.randn(P * T * 7, generator=g)
        self.data = {'cam_pose': torch.randn(T, 4, 4, generator=g), 'cam_pose_inv': torch.randn(T, 4, 4, generator=g), 'person_data': {}}
        for p in range(P):
            self.data['person_data'][p] = {k: torch.randn(T, 26, 3, generator=g) for k in bench.PER_PERSON_OUTPUTS}
        self.scattered = 0

    def _scatter_outputs(self, data):
        self.scattered += 1


def test_dump_writes_every_output_as_float32(bench, tmp_path):
    m = _Model(bench, 2, 30)
    info = bench.dump_outputs(m, m.data, str(tmp_path / 'out'), 0)
    assert m.scattered == 1 and not info['sampled_rows']
    assert sorted(os.listdir(tmp_path / 'out')) == sorted(k + '.npy' for k in ['theta', 'cam_pose', 'cam_pose_inv'] + bench.PER_PERSON_OUTPUTS)
    np.testing.assert_array_equal(np.load(tmp_path / 'out' / 'theta.npy'), m._theta.numpy())
    jw = np.load(tmp_path / 'out' / 'joints_world.npy')
    assert jw.dtype == np.float32 and jw.shape == (60, 26, 3)
    np.testing.assert_array_equal(jw[30:], m.data['person_data'][1]['joints_world'].numpy())


def test_dump_samples_the_same_rows_above_the_limit(bench, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 100_000)
    m = _Model(bench, 3, 40)
    a = bench.dump_outputs(m, m.data, str(tmp_path / 'a'), 0)
    b = bench.dump_outputs(m, m.data, str(tmp_path / 'b'), 0)
    assert a['sampled_rows'] and a['bytes'] <= 100_000
    for k in a['arrays']:
        np.testing.assert_array_equal(np.load(tmp_path / 'a' / (k + '.npy')), np.load(tmp_path / 'b' / (k + '.npy')))
    assert bench.dump_outputs(m, m.data, str(tmp_path / 'c'), 1) is None and not os.path.exists(tmp_path / 'c')


@pytest.mark.gpu
def test_bench_dump_outputs_end_to_end(tmp_path):
    """a short bench run on the GPU writes finite float32 outputs of the 1 x 40 glamr_dynamic problem it timed"""
    out = tmp_path / 'dump'
    r = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--gpus', '1', '--steps', '3', '--warmup', '1', '--frames', '40',
                        '--extras', 'none', '--no-cpu-baseline', '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res['steps'] == 3 and res['outputs_dump']['dir'] == str(out)
    for k in res['outputs_dump']['arrays']:
        a = np.load(out / (k + '.npy'))
        assert a.dtype == np.float32 and np.isfinite(a).all(), k
    assert np.load(out / 'cam_pose.npy').shape == (40, 4, 4)
    assert np.load(out / 'joints_world.npy').shape[0] == 40
