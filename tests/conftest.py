import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

GOLDEN = os.path.join(REPO, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if 'gpu' in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason='no CUDA device'))


@pytest.fixture(scope='session')
def smpl_assets():
    from glamr_b200.synthetic import make_smpl_assets
    return make_smpl_assets(0)
